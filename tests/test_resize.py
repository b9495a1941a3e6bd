"""F5: TransformsUtils.resize_set and FlowsUtils.resize_flow (utils.py:522-560, 107-126) on the sm_100a kernels.

The GPU tests compare bit for bit against the torch port of the reference (oracle/torch_port.py, torch CPU
F.interpolate), values and strides; the backward of the bilinear flow resize against torch CPU autograd.  The
CPU tests check the plug points: what patch() rebinds, and that calls the kernels do not serve reach the
reference's own functions unchanged."""
import contextlib
import sys
import types
from unittest import mock

import numpy as np
import pytest
import torch

import cases
from conftest import load_golden
from master_thesis_b200 import plug
from oracle import torch_port as tp

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def mtb():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device")
    import master_thesis_b200 as m
    from master_thesis_b200 import _lib
    _lib.load()
    return m


def _rand(seed, *shape):
    return torch.from_numpy(np.random.RandomState(seed).random_sample(shape).astype(np.float32))


def _flow(seed, b, f, h, w, planar):
    """A (B,F,h,w,2) flow in one of the two layouts the reference hands over: a contiguous (interleaved) tensor, or
    the permuted view of a planar (B,F,2,h,w) network output (model_dfpn.py:743-744)."""
    t = (_rand(seed, b, f, 2, h, w) * 2 - 1)
    return t.permute(0, 1, 3, 4, 2) if planar else t.permute(0, 1, 3, 4, 2).contiguous()


def _same(got, ref):
    """Same shape, same strides (those of extent-1 dims place nothing and may differ) and bitwise-equal values."""
    assert tuple(got.shape) == tuple(ref.shape)
    st = lambda t: tuple(s if n != 1 else None for s, n in zip(t.stride(), t.shape))   # noqa: E731
    assert st(got) == st(ref), (got.stride(), ref.stride())
    assert torch.equal(got.cpu(), ref), "max |d| = %g" % float((got.cpu() - ref).abs().max())


# ---------------------------------------------------------------- plug points (no GPU)
def _mock_package(resize_set, resize_flow):
    """A ``master_thesis`` stand-in with every class patch() touches; the package re-exports utils' classes."""
    mt = types.ModuleType("master_thesis")
    for mod, cls, attr, _, static in plug._PATCHES:
        m = getattr(mt, mod, None) or types.SimpleNamespace()
        setattr(mt, mod, m)
        k = getattr(m, cls, None) or type(cls, (), {})
        setattr(m, cls, k)
        fn = (lambda *a, **kw: "orig")
        setattr(k, attr, staticmethod(fn) if static else fn)
    mt.utils.TransformsUtils.resize_set = staticmethod(resize_set)
    mt.utils.FlowsUtils.resize_flow = staticmethod(resize_flow)
    mt.TransformsUtils, mt.FlowsUtils = mt.utils.TransformsUtils, mt.utils.FlowsUtils
    return mt


@contextlib.contextmanager
def _patched_package(monkeypatch):
    rs, rf = mock.Mock(return_value="orig_set"), mock.Mock(return_value="orig_flow")
    mt = _mock_package(rs, rf)
    monkeypatch.setitem(sys.modules, "master_thesis", mt)
    names = plug.patch(mt)
    try:
        yield mt, names, rs, rf
    finally:
        plug.unpatch(mt)


def test_patch_rebinds_the_resampling_helpers(monkeypatch):
    with _patched_package(monkeypatch) as (mt, names, rs, rf):
        assert "utils.TransformsUtils.resize_set" in names and "utils.FlowsUtils.resize_flow" in names
        assert mt.TransformsUtils.resize_set is plug.TransformsUtils.resize_set
        assert mt.FlowsUtils.resize_flow is plug.FlowsUtils.resize_flow
    assert mt.TransformsUtils.resize_set is rs and mt.FlowsUtils.resize_flow is rf
    assert "_mt_b200_orig_resize_set" not in mt.TransformsUtils.__dict__


def test_unserved_calls_reach_the_reference(monkeypatch):
    """Host tensors, float64 tensors and modes the kernel does not have go to the saved original, arguments as given."""
    x, v = torch.zeros(1, 3, 2, 8, 8), torch.zeros(1, 1, 2, 8, 8)
    fl = torch.zeros(1, 2, 8, 8, 2)
    with _patched_package(monkeypatch) as (mt, _, rs, rf):
        assert mt.TransformsUtils.resize_set(x, v, x, 4) == "orig_set"
        rs.assert_called_once_with(x, v, x, 4)
        x64 = x.double()
        assert mt.TransformsUtils.resize_set(x64, v.double(), x64, 16) == "orig_set"
        assert rs.call_args.args[0] is x64 and rs.call_args.args[3] == 16
        assert mt.FlowsUtils.resize_flow(fl, (4, 4)) == "orig_flow"
        rf.assert_called_once_with(fl, (4, 4), "nearest")
        assert mt.FlowsUtils.resize_flow(fl.double(), (16, 16), mode="bilinear") == "orig_flow"
        assert mt.FlowsUtils.resize_flow(fl, (16, 16), "bicubic") == "orig_flow"
        assert rf.call_args.args[1:] == ((16, 16), "bicubic")
    plug.unpatch(mt)
    with pytest.raises(RuntimeError, match="no original"):      # a mirror without a saved original never guesses
        plug.TransformsUtils.resize_set(x, v, x, 4)


# ---------------------------------------------------------------- resize_set
def _set_inputs(name):
    if name == "cfg3_like":
        return _rand(1, 2, 3, 5, 256, 256), _rand(2, 2, 1, 5, 256, 256).round(), _rand(3, 2, 3, 5, 256, 256)
    if name == "davis":
        return _rand(4, 1, 3, 2, 480, 854), _rand(5, 1, 1, 2, 480, 854).round(), _rand(6, 1, 3, 2, 480, 854)
    if name == "ragged":
        return _rand(7, 3, 3, 2, 37, 53), _rand(8, 3, 1, 2, 37, 53).round(), _rand(9, 3, 3, 2, 37, 53)
    if name == "sliced":       # x[:, :, 1:4]: strided frames
        x, m, y = _rand(10, 2, 3, 6, 40, 56), _rand(11, 2, 1, 6, 40, 56).round(), _rand(12, 2, 3, 6, 40, 56)
        return x[:, :, 1:4], m[:, :, 1:4], y[:, :, 1:4]
    if name == "frame_major":  # the transposed view of (B,F,C,H,W) memory, as this library writes x_aligned
        x, y = _rand(13, 2, 4, 3, 48, 64).transpose(1, 2), _rand(14, 2, 4, 3, 48, 64).transpose(1, 2)
        return x, _rand(15, 2, 4, 1, 48, 64).round().transpose(1, 2), y
    raise KeyError(name)


SET_CASES = [("cfg3_like", 16), ("cfg3_like", 64), ("davis", 64), ("ragged", 16), ("ragged", 15),
             ("sliced", 16), ("sliced", 64), ("frame_major", 16)]


@gpu
@pytest.mark.parametrize("name,size", SET_CASES)
def test_resize_set_bit_exact(mtb, name, size):
    from master_thesis_b200 import ops
    x, v, y = _set_inputs(name)
    ref = tp.resize_set(x, v, y, size)
    got = ops.resize_set(x.cuda(), v.cuda(), y.cuda(), size)
    for g, r in zip(got, ref):
        _same(g, r)


# ---------------------------------------------------------------- resize_flow
FLOW_CASES = [
    # (name, b, f, h, w, size, mode)
    ("gt_nearest_16", 2, 5, 256, 256, (16, 16), "nearest"),
    ("gt_nearest_64", 2, 5, 256, 256, (64, 64), "nearest"),
    ("bil_16_64", 2, 4, 16, 16, (64, 64), "bilinear"),
    ("bil_64_256", 2, 4, 64, 64, (256, 256), "bilinear"),
    ("bil_256_davis", 1, 2, 256, 256, (480, 854), "bilinear"),
    ("bil_down_ragged", 2, 3, 37, 53, (16, 13), "bilinear"),
    ("near_up_ragged", 2, 3, 13, 7, (21, 11), "nearest"),
]


@gpu
@pytest.mark.parametrize("planar", [False, True], ids=["interleaved", "planar"])
@pytest.mark.parametrize("name,b,f,h,w,size,mode", FLOW_CASES)
def test_resize_flow_bit_exact(mtb, name, b, f, h, w, size, mode, planar):
    from master_thesis_b200 import ops
    fl = _flow(sum(map(ord, name)), b, f + 1, h, w, planar)
    if name.startswith("gt_"):         # flow_gt[:, r_list] (model_dfpn.py:354-355): advanced indexing
        r_list = [i for i in range(f + 1) if i != (f + 1) // 2]
        src, dsrc = fl[:, r_list], fl.cuda()[:, r_list]
    else:                              # a frame slice: for b > 1 the reference's reshape copies (interleaved result)
        src, dsrc = fl[:, 1:], fl.cuda()[:, 1:]
        _same(ops.resize_flow(fl.cuda(), size, mode), tp.resize_flow(fl, size, mode))
    _same(ops.resize_flow(dsrc, size, mode), tp.resize_flow(src, size, mode))


BWD_CASES = [("bil_16_64", 2, 4, 16, 16, (64, 64)), ("bil_64_256", 2, 4, 64, 64, (256, 256)),
             ("bil_256_davis", 1, 2, 256, 256, (480, 854)), ("bil_down_ragged", 2, 3, 37, 53, (16, 13))]


@gpu
@pytest.mark.parametrize("name,b,f,h,w,size", BWD_CASES)
def test_resize_flow_backward(mtb, name, b, f, h, w, size):
    """d loss / d flow of the bilinear resize against torch CPU autograd; the gather is deterministic."""
    from master_thesis_b200 import ops
    fl = _flow(sum(map(ord, name)) + 1, b, f, h, w, True)
    wgt = _rand(99, b, f, size[0], size[1], 2) - 0.5
    ref_in = fl.clone().requires_grad_(True)
    (tp.resize_flow(ref_in, size, "bilinear") * wgt).sum().backward()
    grads = []
    for _ in range(2):
        d = fl.cuda().requires_grad_(True)
        (ops.resize_flow(d, size, "bilinear") * wgt.cuda()).sum().backward()
        grads.append(d.grad.cpu())
    ref = ref_in.grad
    assert tuple(grads[0].shape) == tuple(ref.shape)
    assert float((grads[0] - ref).abs().max()) <= 1e-5 * float(ref.abs().max())
    assert torch.equal(grads[0], grads[1])


# ---------------------------------------------------------------- guard bands
@gpu
def test_resize_no_out_of_bounds_writes(mtb):
    """Every output is carved out of a sentinel-filled buffer; the guard bands around it must be untouched after the
    calls.  Ragged shapes: partial 4-pixel chunks, sizes that are not multiples of 4, both flow layouts."""
    from master_thesis_b200 import _lib, ops
    G = 256
    made = []

    def guarded_empty(*a, **k):
        probe = torch.empty(*a, **{**k, "device": "meta"})
        n = probe.numel()
        buf = torch.full((n + 2 * G,), -12345.0, dtype=probe.dtype, device=k.get("device", "cuda"))
        made.append((buf, n))
        return _lib.keep(buf[G:G + n].view(probe.shape))

    orig, orig_like = ops._empty, ops._empty_like
    ops._empty = guarded_empty
    ops._empty_like = lambda t, **k: guarded_empty(t.shape, dtype=t.dtype, device=t.device)
    try:
        x, v, y = (t.cuda() for t in _set_inputs("ragged"))
        for size in (15, 16, 17, 64):
            ops.resize_set(x, v, y, size)
        for planar in (False, True):
            fl = _flow(3, 2, 3, 13, 7, planar).cuda()
            for size in ((21, 11), (6, 5), (64, 64)):
                ops.resize_flow(fl, size, "nearest")
                d = fl.clone().requires_grad_(True)
                ops.resize_flow(d, size, "bilinear").sum().backward()
        torch.cuda.synchronize()
    finally:
        ops._empty, ops._empty_like = orig, orig_like
    assert len(made) >= 30
    for buf, n in made:
        assert bool((buf[:G] == -12345.0).all()) and bool((buf[G + n:] == -12345.0).all()), \
            "guard band overwritten (n=%d)" % n


# ---------------------------------------------------------------- plug points on the GPU
@gpu
def test_mirrors_route_by_what_the_kernels_serve(mtb, monkeypatch):
    x, v, y = (t.cuda() for t in _set_inputs("ragged"))
    fl = _flow(4, 2, 3, 16, 16, True).cuda()
    with _patched_package(monkeypatch) as (mt, _, rs, rf):
        _same(mt.TransformsUtils.resize_set(x, v, y, 16)[0], tp.resize_set(x.cpu(), v.cpu(), y.cpu(), 16)[0])
        _same(mt.FlowsUtils.resize_flow(fl, (64, 64), "bilinear"), tp.resize_flow(fl.cpu(), (64, 64), "bilinear"))
        assert not rs.called and not rf.called
        xg = x.clone().requires_grad_(True)
        assert mt.TransformsUtils.resize_set(xg, v, y, 16) == "orig_set"            # a gradient: no kernel for it
        assert mt.TransformsUtils.resize_set(x.double(), v.double(), y.double(), 16) == "orig_set"
        assert mt.FlowsUtils.resize_flow(fl, (64, 64), "bicubic") == "orig_flow"
        assert mt.FlowsUtils.resize_flow(fl.clone().requires_grad_(True), (64, 64)) == "orig_flow"   # nearest + grad
        assert rs.call_count == 2 and rf.call_count == 2


@gpu
@pytest.mark.parametrize("name", sorted(cases.DFPNLOSS_CASES))
def test_dfpn_training_step_with_resize_kernels(mtb, name):
    """plug.dfpn_train_val_wrapper + dfpn_compute_loss with the resampling mirrors behind the package's
    TransformsUtils / FlowsUtils: the goldens of the unmodified reference at the tolerances of the torch-port run,
    and the recorded plan now holds the resize launches."""
    from master_thesis_b200 import _lib
    spec = cases.DFPNLOSS_CASES[name]
    x, m, y, flow_gt, use, corr, f16, f64, fhw, feats = cases.dfpnloss_inputs(spec)
    g = load_golden("dfpnloss_" + name)
    n = x.shape[2]
    t, r_list = n // 2, [i for i in range(n) if i != n // 2]
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()   # noqa: E731
    leaves = [dev(a).requires_grad_(True) for a in (corr, f16, f64, fhw)]

    class _DFPNLike(object):
        def __call__(self, *a):
            return tuple(leaves)

        def model_vgg(self, inp):
            return [None, None, None, dev(feats)]

    stub = types.ModuleType("master_thesis")
    stub.TransformsUtils = types.SimpleNamespace(resize_set=plug.TransformsUtils.resize_set)
    stub.FlowsUtils = types.SimpleNamespace(resize_flow=plug.FlowsUtils.resize_flow)
    saved = sys.modules.get("master_thesis")
    sys.modules["master_thesis"] = stub
    try:
        fake = _DFPNLike()
        with _lib.record() as plan:
            res = plug.dfpn_train_val_wrapper(fake, dev(x), dev(m), dev(y), dev(flow_gt), dev(use), t, r_list)
            loss, items = plug.dfpn_compute_loss(fake, *res, t, r_list)
            grads = torch.autograd.grad(loss, leaves)
    finally:
        if saved is None:
            del sys.modules["master_thesis"]
        else:
            sys.modules["master_thesis"] = saved
    assert sorted(plan.names()) == sorted(["mt_resize_set"] * 2 + ["mt_resize_flow"] * 2 +
                                          ["mt_corr4d_vgg_l1_fwd", "mt_corr4d_l1_bwd"] + ["mt_masked_l1_fwd"] * 3 +
                                          ["mt_warp_l1_fwd"] * 2 + ["mt_warp_l1_bwd"] * 2 + ["mt_masked_l1_bwd"] * 3)
    # the resized sets and ground-truth flows equal the reference's
    xc, mc, yc, fc = (torch.from_numpy(a) for a in (x, m, y, flow_gt))
    for got, ref in zip(res[1][:2] + res[2][:2] + res[3][:2],
                        [tp.resize_set(xc, 1 - mc, yc, s)[k] for k in range(3) for s in (16, 64)]):
        _same(got, ref)
    for got, s in zip(res[6][:2], (16, 64)):
        _same(got, tp.resize_flow(fc[:, r_list], (s, s)))
    assert abs(float(items[0]) - float(g["items"][0])) <= 1e-3
    assert float(loss) - float(items[0]) == pytest.approx(float(g["loss"]) - float(g["items"][0]), rel=1e-5)
    assert np.allclose([float(i) for i in items[1:]], g["items"][1:], rtol=1e-5, atol=0)
    assert np.abs(grads[2].cpu().numpy() - g["g_flow64"]).max() <= 2e-5 * np.abs(g["g_flow64"]).max()
    assert np.abs(grads[3].cpu().numpy() - g["g_flowhw"]).max() <= 2e-5 * np.abs(g["g_flowhw"]).max()
    assert float(grads[1].abs().double().sum()) == pytest.approx(float(g["g_flow16_abs"]), rel=1e-5)
    assert float(grads[0].abs().double().sum()) == pytest.approx(float(g["g_corr_abs"]), rel=1e-3)
