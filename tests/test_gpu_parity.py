"""GPU parity tests: the sm_100a kernels (through the C ABI and the plug-point
mirrors) against the CPU oracle and the reference's golden vectors.

Bar (BASELINE.json north_star): index / mask logic bit-exact; fp32 warp /
composite within 1e-5 abs (the kernels follow the reference's CPU operation
order, so most are in fact bit-exact and asserted as such); reductions within
1e-5 relative; correlation within 1e-2 relative when it runs on tensor cores
(TF32), 2e-6 abs on the fp32 SIMT path.
"""
import numpy as np
import pytest
import torch

import cases
import oracle
from conftest import load_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mtb():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device")
    import master_thesis_b200 as m
    from master_thesis_b200 import _lib
    _lib.load()
    return m


def dev(a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.detach().contiguous().cpu().numpy()


# ---------------------------------------------------------------- a1 / a2
@pytest.mark.parametrize("name", sorted(cases.WARP_CASES))
def test_dfpn_align_tail(mtb, name):
    x, m, m_t, flow = cases.warp_inputs(cases.WARP_CASES[name])
    g = load_golden("warp_" + name)
    xa, va, vm = mtb.dfpn_align_tail(dev(x), dev(m), dev(m_t), dev(flow))
    assert xa.shape == x.shape and va.shape == m.shape and vm.shape == m.shape
    # same strides as the reference's transposed view (utils.py:97)
    b, c, f, h, w = x.shape
    assert xa.stride() == (f * c * h * w, h * w, c * h * w, w, 1)
    oxa, ova, ovm = oracle.dfpn_align_tail(x, m, m_t, flow)
    for got, orc, gold in ((xa, oxa, g["x_aligned"]), (va, ova, g["v_aligned"]), (vm, ovm, g["v_map"])):
        got = host(got)
        assert np.array_equal(got, orc)
        assert np.array_equal(got, gold)


@pytest.mark.parametrize("name", ["smooth_f4", "f1_odd"])
def test_align_set_plug_and_views(mtb, name):
    x, m, m_t, flow = cases.warp_inputs(cases.WARP_CASES[name])
    g = load_golden("warp_" + name)
    b, c, f, h, w = x.shape
    # non-contiguous inputs: slices of a larger clip, like x[:, :, r_list] views
    big = torch.zeros((b, c, f + 2, h, w), device="cuda")
    big[:, :, 1:f + 1] = dev(x)
    vbig = torch.zeros((b, 1, f + 2, h, w), device="cuda")
    vbig[:, :, 1:f + 1] = dev(1 - m)
    xa, va = mtb.FlowsUtils.align_set(big[:, :, 1:f + 1], vbig[:, :, 1:f + 1], dev(flow))
    assert np.array_equal(host(xa), g["x_aligned"])
    assert np.array_equal(host(va), g["v_aligned"])


def test_warp_rejects_cpu_tensors(mtb):
    with pytest.raises(RuntimeError):
        mtb.FlowsUtils.align_set(torch.zeros(1, 3, 1, 4, 4), torch.zeros(1, 1, 1, 4, 4),
                                 torch.zeros(1, 1, 4, 4, 2))


# ---------------------------------------------------------------- a3
@pytest.mark.parametrize("name", sorted(cases.CPN_CASES))
def test_cpn_align_tail(mtb, name):
    x, m, m_t, theta = cases.cpn_inputs(cases.CPN_CASES[name])
    g = load_golden("cpn_" + name)
    # theta mode: bit-exact against the oracle (same scalar linspace algorithm) ...
    xa, va, vm = mtb.cpn_align_tail(dev(x), dev(m), dev(m_t), dev(theta))
    oxa, ova, ovm = oracle.cpn_align_tail(x, m, m_t, theta=theta)
    assert np.array_equal(host(xa), oxa)
    assert np.array_equal(host(va), ova)
    assert np.array_equal(host(vm), ovm)
    # ... and within tolerance of the reference (its vectorised linspace differs by 1 ulp)
    assert np.abs(host(xa) - g["x_aligned"]).max() <= 1e-5
    bad = host(va) != g["v_aligned"]
    assert np.all(np.abs(g["v_soft"][bad] - 0.5) <= 1e-5) and bad.mean() <= 2e-3
    # dense-grid mode with the reference's own grid: bit-exact against the reference
    from master_thesis_b200 import ops
    xa, va, vm = ops.warp_fwd(dev(x), dev(m), dev(g["grid"]), dev(m_t),
                              ops.VIS_BILINEAR | ops.VIS_FROM_MASK)
    assert np.array_equal(host(xa), g["x_aligned"])
    assert np.array_equal(host(va), g["v_aligned"])
    assert np.array_equal(host(vm), g["v_map"])


# Sizes that engage the persistent TMA-staged kernel (warp_tma.cu: >= 2 tiles per SM); the
# golden cases above are small and take the direct-gather kernel.
STAGED_CASES = {
    # partial tiles on both axes, moderate thetas: almost every tile staged
    "rand": dict(seed=71, b=3, f=4, h=200, w=204, sigma=0.1),
    # large thetas: most footprints exceed the box -> in-kernel direct path, out-of-frame taps
    "big": dict(seed=72, b=2, f=4, h=224, w=208, sigma=0.6),
    # near-identity: every tile staged, border tiles exercise the zero-padded visibility
    "ident": dict(seed=73, b=4, f=2, h=256, w=256, sigma=0.01),
    # exact half-pixel translations: the soft visibility lands exactly on 0.5 (strict >)
    "halfpix": dict(seed=74, b=2, f=4, h=192, w=256, sigma=0.0),
}


def _set_tuning(name, value):
    from master_thesis_b200 import _lib
    _lib.call("mt_set_tuning", name.encode(), value)


@pytest.mark.parametrize("name", sorted(STAGED_CASES))
def test_cpn_align_tail_staged(mtb, name):
    """The staged kernel against the oracle and the direct kernel."""
    spec = STAGED_CASES[name]
    x, m, m_t, theta = cases.cpn_inputs(spec)
    oxa, ova, ovm = oracle.cpn_align_tail(x, m, m_t, theta=theta)
    try:
        _set_tuning("MT_WARP_STAGED", 1)
        xa, va, vm = mtb.cpn_align_tail(dev(x), dev(m), dev(m_t), dev(theta))
        _set_tuning("MT_WARP_STAGED", 0)
        xd, vd, vmd = mtb.cpn_align_tail(dev(x), dev(m), dev(m_t), dev(theta))
    finally:
        _set_tuning("MT_WARP_STAGED", 1)
    for got, direct, orc in ((xa, xd, oxa), (va, vd, ova), (vm, vmd, ovm)):
        assert np.array_equal(host(got), orc)           # staged kernel == oracle, bit for bit
        assert np.array_equal(host(direct), orc)        # direct-gather kernel == oracle
    b, c, f, h, w = x.shape
    assert xa.stride() == (f * c * h * w, h * w, c * h * w, w, 1)


def test_cpn_align_tail_staged_views(mtb):
    """Strided inputs (x[:, :, r_list]-style slices of a longer clip) through the TMA maps."""
    spec = STAGED_CASES["rand"]
    x, m, m_t, theta = cases.cpn_inputs(spec)
    b, c, f, h, w = x.shape
    big = torch.full((b, c, f + 3, h, w), 7.0, device="cuda")
    big[:, :, 2:f + 2] = dev(x)
    mbig = torch.full((b, 1, f + 3, h, w), 1.0, device="cuda")
    mbig[:, :, 2:f + 2] = dev(m)
    xa, va, vm = mtb.cpn_align_tail(big[:, :, 2:f + 2], mbig[:, :, 2:f + 2], dev(m_t), dev(theta))
    oxa, ova, ovm = oracle.cpn_align_tail(x, m, m_t, theta=theta)
    assert np.array_equal(host(xa), oxa) and np.array_equal(host(va), ova) and np.array_equal(host(vm), ovm)


class _FakeCPN(object):
    def __init__(self, theta):
        self.theta = theta

    def A_Encoder(self, xx, mm):
        return torch.zeros(xx.size(0), 1, 1, 1, device=xx.device)

    def A_Regressor(self, a, b):
        return self.theta


class _FakeDFPN(object):
    def __init__(self, flow):
        self.flow = flow

    def __call__(self, *a):
        return None, None, None, self.flow


def test_aligner_protocol_mirrors(mtb):
    """DFPN.align / CPN.align replacements with the CNNs stubbed, as in make_golden.py."""
    x, m, m_t, theta = cases.cpn_inputs(cases.CPN_CASES["rand_f4"])
    xa, va, vm = mtb.cpn_align(_FakeCPN(dev(theta)), dev(x[:, :, 0]), dev(m_t), dev(x), dev(m))
    oxa, ova, ovm = oracle.cpn_align_tail(x, m, m_t, theta=theta)
    assert np.array_equal(host(xa), oxa) and np.array_equal(host(va), ova) and np.array_equal(host(vm), ovm)
    x, m, m_t, flow = cases.warp_inputs(cases.WARP_CASES["smooth_f4"])
    g = load_golden("warp_smooth_f4")
    xa, va, vm = mtb.dfpn_align(_FakeDFPN(dev(flow)), dev(x[:, :, 0]), dev(m_t), dev(x), dev(m))
    assert np.array_equal(host(xa), g["x_aligned"]) and np.array_equal(host(vm), g["v_map"])


# ---------------------------------------------------------------- a4 / a5 / a6
@pytest.mark.parametrize("name", sorted(cases.LOSS_CASES))
def test_losses_and_backward(mtb, name):
    x, m, flow, flow_gt, use, t, r_list = cases.loss_inputs(cases.LOSS_CASES[name])
    g = load_golden("loss_" + name)
    f = len(r_list)
    xt, vt = dev(x), dev(1 - m)
    fl = dev(flow).requires_grad_(True)
    mo = mtb.LossesUtils.mask_out(fl)
    assert np.array_equal(host(mo), g["mask_out"])
    # the reference's own sequence (model_dfpn.py:377-383, 269-287) on the patched ops
    xa, va = mtb.FlowsUtils.align_set(xt[:, :, r_list], vt[:, :, r_list], fl)
    y_hat = xt[:, :, t].unsqueeze(2).repeat(1, 1, f, 1, 1)
    mask = vt[:, :, t].unsqueeze(2).repeat(1, 1, f, 1, 1) * (1 - mo)
    rec = mtb.LossesUtils.masked_l1(y_hat, xa, mask, reduction='sum')
    assert float(rec) == pytest.approx(float(g["recons"]), rel=1e-5)
    g_xa, = torch.autograd.grad(rec, xa, retain_graph=True)
    scale = np.abs(g["g_x_aligned"]).max()
    assert np.abs(host(g_xa) - g["g_x_aligned"]).max() <= 1e-5 * scale
    g_fl, = torch.autograd.grad(rec, fl)
    gscale = np.abs(g["g_flow"]).max()
    assert np.abs(host(g_fl) - g["g_flow"]).max() <= 2e-5 * gscale
    mean = mtb.LossesUtils.masked_l1(y_hat, xa.detach(), mask, reduction='mean', weight=2)
    assert float(mean) == pytest.approx(float(g["mean_l1"]), rel=1e-5)
    # flow L1 with batch selection (model_dfpn.py:259-267), no host sync
    fl1 = mtb.LossesUtils.masked_l1(fl, dev(flow_gt), torch.ones_like(fl), dev(use.astype(np.uint8)))
    assert float(fl1) == pytest.approx(float(g["flow_l1"]), rel=1e-5)
    g_fl1, = torch.autograd.grad(fl1, fl)
    assert np.abs(host(g_fl1) - g["g_flow_l1"]).max() <= 1e-6 * np.abs(g["g_flow_l1"]).max() + 1e-12
    none = mtb.LossesUtils.masked_l1(fl, dev(flow_gt), torch.ones_like(fl),
                                     torch.zeros(len(use), dtype=torch.bool))
    assert float(none) == 0.0
    # fused one-pass form (K1c): same loss, same flow gradient
    fl2 = dev(flow).requires_grad_(True)
    fused = mtb.LossesUtils.alignment_recons(xt[:, :, t], vt[:, :, t], xt[:, :, r_list],
                                             vt[:, :, r_list], fl2)
    assert float(fused) == pytest.approx(float(g["recons"]), rel=1e-5)
    fused.backward()
    assert np.abs(host(fl2.grad) - g["g_flow"]).max() <= 2e-5 * gscale
    # fused + materialised outputs
    from master_thesis_b200 import ops
    loss, xa2, va2 = ops.warp_masked_l1(xt[:, :, r_list], vt[:, :, r_list], dev(flow), xt[:, :, t],
                                        vt[:, :, t], materialize=True)
    assert np.array_equal(host(xa2), host(xa)) and np.array_equal(host(va2), host(va))
    assert float(loss) == pytest.approx(float(g["recons"]), rel=1e-5)


# ---------------------------------------------------------------- a7
def _corr_tol_check(c, g, spec, tc):
    if tc:   # TF32 operands, fp32 accumulate: north_star tolerance <= 1e-2 relative; cosine values are <= 1
        cases.corr_check(c, g, spec, 2e-3)
    else:
        cases.corr_check(c, g, spec, 2e-6)


@pytest.mark.parametrize("name", sorted(cases.CORR_CASES))
def test_corr4d(mtb, name):
    from master_thesis_b200 import _lib
    spec = cases.CORR_CASES[name]
    ft, vt, fr, vr = cases.corr_inputs(spec)
    g = load_golden("corr_" + name)
    c = host(mtb.CorrelationVGG.correlation_masked_4d(dev(ft), dev(vt), dev(fr), dev(vr)))
    tc = _lib.load().mt_corr4d_uses_tensor_cores(spec["c"], spec["h"] * spec["w"])
    _corr_tol_check(c, g, spec, tc)
    if vt is not None:       # masked rows are exactly zero
        assert np.all(c[0, :, 0, :] == 0.0)


@pytest.mark.parametrize("tm", [256, 128])
@pytest.mark.parametrize("tn", [64, 128, 256])
@pytest.mark.parametrize("name", ["real_masked", "real_nomask", "mid_masked", "big_masked"])
def test_corr4d_every_tile_variant(mtb, name, tn, tm):
    """Every corr_tc_kernel instantiation (128 / 256 output rows x 64 / 128 / 256 output columns per CTA: different
    accumulator halves, epilogue offsets, scale tables, norm-warp mappings, stage counts and grids) on small, medium
    (40 frames) and cfg3-size (128 frames) batches, against the golden vectors of the reference AND the whole
    volume of the CPU oracle."""
    spec = cases.CORR_CASES[name]
    ft, vt, fr, vr = cases.corr_inputs(spec)
    g = load_golden("corr_" + name)
    try:
        _set_tuning("MT_CORR_TN", tn)
        _set_tuning("MT_CORR_TM", tm)
        c = host(mtb.CorrelationVGG.correlation_masked_4d(dev(ft), dev(vt), dev(fr), dev(vr)))
    finally:
        _set_tuning("MT_CORR_TN", 0)
        _set_tuning("MT_CORR_TM", 0)
    _corr_tol_check(c, g, spec, True)
    o = oracle.corr4d(ft, vt, fr, vr)
    err = np.abs(c - o)
    assert err.max() <= 2e-3 and err.max() <= 1e-2 * np.abs(o).max()
    if vt is not None:       # masked rows / columns are exactly zero in every frame
        assert np.array_equal(c == 0.0, o == 0.0)


@pytest.mark.parametrize("tn", [128, 256])
@pytest.mark.parametrize("name", ["real_masked", "real_nomask", "mid_masked", "big_masked"])
def test_corr4d_cta_pairs(mtb, name, tn):
    """The CTA-pair kernel (tcgen05 cta_group::2: M = 256 over two SMs, each CTA stages its half of A and of B,
    column scales exchanged through distributed shared memory) on 2 / 40 / 128 frames: more tiles than pairs, fewer
    tiles than pairs, masked and unmasked - against the reference's golden vectors and the whole oracle volume."""
    spec = cases.CORR_CASES[name]
    ft, vt, fr, vr = cases.corr_inputs(spec)
    g = load_golden("corr_" + name)
    try:
        _set_tuning("MT_CORR_2CTA", 1)
        _set_tuning("MT_CORR_TN", tn)
        c = host(mtb.CorrelationVGG.correlation_masked_4d(dev(ft), dev(vt), dev(fr), dev(vr)))
    finally:
        _set_tuning("MT_CORR_TN", 0)
        _set_tuning("MT_CORR_2CTA", -1)
    _corr_tol_check(c, g, spec, True)
    o = oracle.corr4d(ft, vt, fr, vr)
    err = np.abs(c - o)
    assert err.max() <= 2e-3 and err.max() <= 1e-2 * np.abs(o).max()
    if vt is not None:
        assert np.array_equal(c == 0.0, o == 0.0)


def test_corr4d_large_batch_takes_cta_pairs(mtb):
    """384 frames (B = 96, F = 4): the default heuristic hands the batch to the CTA-pair kernel (5.2 whole-frame tiles
    per pair).  Compared with the single-CTA kernel on the whole volume and with the CPU oracle on the first and the
    last two samples."""
    from master_thesis_b200 import ops, synth
    ft, vt, fr, vr = synth.vgg_feats(23, 96, 4)
    dft, dvt, dfr, dvr = dev(ft), dev(vt), dev(fr), dev(vr)
    c_pair = host(ops.corr4d(dft, dvt, dfr, dvr))
    try:
        _set_tuning("MT_CORR_2CTA", 0)
        c_one = host(ops.corr4d(dft, dvt, dfr, dvr))
    finally:
        _set_tuning("MT_CORR_2CTA", -1)
    assert np.abs(c_pair - c_one).max() <= 1e-4          # same TF32 products, different accumulation order
    assert np.array_equal(c_pair == 0.0, c_one == 0.0)
    for sl in (slice(0, 2), slice(94, 96)):
        o = oracle.corr4d(ft[sl], vt[sl], fr[sl], vr[sl])
        assert np.abs(c_pair[sl] - o).max() <= 2e-3 and np.array_equal(c_pair[sl] == 0.0, o == 0.0)


# ---------------------------------------------------------------- a8
@pytest.mark.parametrize("table", [2, 1, 0])
@pytest.mark.parametrize("name", sorted(cases.CM_CASES))
def test_cm_module(mtb, name, table):
    """table=2: masks | one grouped launch for similarity + softmax table + copy (default: c_feats crosses HBM once);
    table=1: masks | similarity | copy with the softmax looked up per mask pattern;
    table=0: the separate per-pixel weights kernel (the path 8 references take)."""
    from master_thesis_b200 import ops
    cf, vt, va = cases.cm_inputs(cases.CM_CASES[name])
    g = load_golden("cm_" + name)
    oout, ocmask, ogs = oracle.cm_module(cf, vt, va, return_gs=True)
    try:
        _set_tuning("MT_CM_TABLE", table)
        out, cmask = mtb.CM_Module()(dev(cf), dev(vt), dev(va))
        out, cmask = host(out), host(cmask)
        _, _, gs = ops.cm_match(dev(cf), dev(vt), dev(va), return_gs=True)
        gs = gs.clone()
    finally:
        _set_tuning("MT_CM_TABLE", 2)
    assert np.abs(host(gs) - ogs).max() <= 1e-6 * max(1.0, np.abs(ogs).max())
    assert np.abs(out - oout).max() <= 1e-5 and np.abs(cmask - ocmask).max() <= 2e-6
    assert np.abs(cmask - g["c_mask"]).max() <= 2e-6
    if "out" in g:
        assert np.abs(out - g["out"]).max() <= 1e-5
    else:
        assert np.abs(out.reshape(-1)[::53] - g["sample"]).max() <= 1e-5


@pytest.mark.parametrize("shape", [(5, 4, 9, 24, 48), (3, 2, 5, 32, 32), (9, 5, 16, 16, 80), (1, 8, 6, 16, 16),
                                   (2, 9, 7, 16, 24)])
def test_cm_ragged(mtb, shape):
    """All three launch structures against the oracle on shapes that leave partial 1024-pixel chunks, a channel
    count that is not a multiple of the slab, one sample, and 1 / 3 / 4 / 7 / 8 references (8: the grouped and the
    table variants fall back to the weights kernel)."""
    from master_thesis_b200 import ops, synth
    b, f, c, h, w = shape
    cf, vt, va = synth.cm_inputs(61 + b, b, f, c, h, w, 4)
    oout, ocm, ogs = oracle.cm_module(cf, vt, va, return_gs=True)
    res = {}
    try:
        for table in (2, 1, 0):
            _set_tuning("MT_CM_TABLE", table)
            out, cmask, gs = ops.cm_match(dev(cf), dev(vt), dev(va), return_gs=True)
            res[table] = (host(out), host(cmask), host(gs.clone()))
    finally:
        _set_tuning("MT_CM_TABLE", 2)
    for table in (2, 1, 0):
        out, cmask, gs = res[table]
        assert np.abs(gs - ogs).max() <= 1e-6 * max(1.0, np.abs(ogs).max())
        assert np.abs(out - oout).max() <= 1e-5 and np.abs(cmask - ocm).max() <= 2e-6
    # same partial sums folded in a different (fixed) order: the two paths agree to rounding
    assert np.abs(res[1][0] - res[0][0]).max() <= 1e-5 and np.abs(res[1][1] - res[0][1]).max() <= 2e-6
    assert np.abs(res[2][0] - res[1][0]).max() <= 1e-5 and np.abs(res[2][1] - res[1][1]).max() <= 2e-6


@pytest.mark.parametrize("groups", [1, 2, 3, 64])
def test_cm_grouped_rounds(mtb, groups):
    """The grouped single-launch kernel with fewer groups than samples (a group then walks several samples:
    B = 5 in rounds of 1 / 2 / 3) and with more groups requested than samples (clamped to B)."""
    from master_thesis_b200 import ops, synth
    b, f, c, h, w = 5, 5, 24, 32, 40
    cf, vt, va = synth.cm_inputs(77, b, f, c, h, w, 4)
    va[1] = 0.0                      # one sample without any visible reference pixel (v_sum guard)
    oout, ocm, ogs = oracle.cm_module(cf, vt, va, return_gs=True)
    try:
        _set_tuning("MT_CM_TABLE", 2)
        _set_tuning("MT_CM_GROUPS", groups)
        for rep in range(2):          # twice: the arrival counters are re-armed by the masks kernel of every call
            out, cmask, gs = ops.cm_match(dev(cf), dev(vt), dev(va), return_gs=True)
            out, cmask, gs = host(out), host(cmask), host(gs.clone())
            assert np.abs(gs - ogs).max() <= 1e-6 * max(1.0, np.abs(ogs).max())
            assert np.abs(out - oout).max() <= 1e-5 and np.abs(cmask - ocm).max() <= 2e-6
    finally:
        _set_tuning("MT_CM_GROUPS", 0)


@pytest.mark.parametrize("keep", [8, 1, 0])
def test_cm_grouped_full_size(mtb, keep):
    """cfg2 size (B = 8, 128 x 5 x 64 x 64: 14 items per CTA) so that pass 2 of the grouped kernel takes its
    operands from all three places: the last batch from registers, `keep` batches from shared memory, the rest
    from L2.  Checked against the oracle and against the two-launch form."""
    from master_thesis_b200 import ops, synth
    cf, vt, va = synth.cm_inputs(91, 8, 5, 128, 64, 64)
    oout, ocm, ogs = oracle.cm_module(cf, vt, va, return_gs=True)
    dcf, dvt, dva = dev(cf), dev(vt), dev(va)
    try:
        _set_tuning("MT_CM_KEEP", keep)
        out, cmask, gs = ops.cm_match(dcf, dvt, dva, return_gs=True)
        out, cmask, gs = host(out), host(cmask), host(gs.clone())
        _set_tuning("MT_CM_TABLE", 1)
        out1, cmask1 = ops.cm_match(dcf, dvt, dva)
        out1, cmask1 = host(out1), host(cmask1)
    finally:
        _set_tuning("MT_CM_KEEP", 0)
        _set_tuning("MT_CM_TABLE", 2)
    assert np.abs(gs - ogs).max() <= 1e-6 * max(1.0, np.abs(ogs).max())
    assert np.abs(out - oout).max() <= 1e-5 and np.abs(cmask - ocm).max() <= 2e-6
    assert np.array_equal(out[:, :128], cf[:, :, 0].reshape(8, 128, 64, 64))      # cat[c_t, ...]: a plain copy
    assert np.abs(out - out1).max() <= 1e-5 and np.abs(cmask - cmask1).max() <= 2e-6


@pytest.mark.parametrize("world", [2, 3, 8])
def test_sharded_launches_equal_unsharded(mtb, world):
    """SURVEY 8(e) on the GPU: the (b, f) blocks of shard.frame_shard_groups (strided views of the full tensors,
    one launch per group) and the per-sample CM shards of shard.batch_shard reproduce the unsharded launch bit
    for bit - every emulated rank runs in turn on this GPU; there is no data-path collective to test."""
    from master_thesis_b200 import ops, shard, synth
    x, m, m_t, flow = cases.warp_inputs(cases.WARP_CASES["smooth_f4"])
    b, c, f, h, w = x.shape
    dx, dm, dmt, dfl = dev(x), dev(m), dev(m_t), dev(flow)
    theta = dev(synth.thetas(5, b * f, 0.1))
    full_d = [host(t) for t in mtb.dfpn_align_tail(dx, dm, dmt, dfl)]
    full_c = [host(t) for t in mtb.cpn_align_tail(dx, dm, dmt, theta)]
    got_d = [np.zeros_like(t) for t in full_d]
    got_c = [np.zeros_like(t) for t in full_c]
    owned = np.zeros((b, f), np.int32)
    for rank in range(world):
        for bi, (f0, f1) in shard.frame_shard_groups(b, f, rank, world).items():
            owned[bi, f0:f1] += 1
            part = mtb.dfpn_align_tail(dx[bi:bi + 1, :, f0:f1], dm[bi:bi + 1, :, f0:f1], dmt[bi:bi + 1], dfl[bi:bi + 1, f0:f1])
            for dst, src in zip(got_d, part):
                dst[bi, :, f0:f1] = host(src)[0]
            th = theta.view(b, f, 2, 3)[bi, f0:f1].reshape(-1, 2, 3)
            part = mtb.cpn_align_tail(dx[bi:bi + 1, :, f0:f1], dm[bi:bi + 1, :, f0:f1], dmt[bi:bi + 1], th)
            for dst, src in zip(got_c, part):
                dst[bi, :, f0:f1] = host(src)[0]
    assert np.all(owned == 1)                        # the shards tile the B x F range exactly once
    for a_, b_ in zip(got_d + got_c, full_d + full_c):
        assert np.array_equal(a_, b_)
    cf, vt, va = cases.cm_inputs(cases.CM_CASES["edge"])
    dcf, dvt, dva = dev(cf), dev(vt), dev(va)
    out, cmask = [host(t) for t in ops.cm_match(dcf, dvt, dva)]
    for rank in range(world):
        lo, hi = shard.batch_shard(cf.shape[0], rank, world)
        if hi > lo:
            o, cm = ops.cm_match(dcf[lo:hi], dvt[lo:hi], dva[lo:hi])
            # a sample's result depends on its batch only through the number of CTAs that share its partial sums
            assert np.abs(host(o) - out[lo:hi]).max() <= 1e-6 and np.abs(host(cm) - cmask[lo:hi]).max() <= 2e-6


# ---------------------------------------------------------------- a9 .. a12
class _FakeCHN(object):
    def __init__(self, nn_out):
        self.nn_out = nn_out
        self.seen = None

    def nn(self, inp):
        self.seen = inp
        return self.nn_out


@pytest.mark.parametrize("name", sorted(cases.CHN_CASES))
def test_chn(mtb, name):
    from master_thesis_b200 import ops
    x_t, v_t, x_al, v_al, v_map, nn_out = cases.chn_inputs(cases.CHN_CASES[name])
    g = load_golden("chn_" + name)
    b, _, f, h, w = x_al.shape
    fake = _FakeCHN(dev(nn_out).requires_grad_(True))
    y_hat, y_comp = mtb.chn_forward(fake, dev(x_t), dev(v_t), dev(x_al), dev(v_al), dev(v_map))
    assert np.array_equal(host(fake.seen), g["nn_input"])
    assert y_hat.shape == (b, 3, f, h, w)
    assert np.array_equal(host(y_hat), g["y_hat"])
    assert np.array_equal(host(y_comp), g["y_hat_comp"])
    r = cases.synth.rng(cases.CHN_CASES[name]["seed"] + 7)
    gy = r.standard_normal(y_hat.shape).astype(np.float32)
    gc = r.standard_normal(y_hat.shape).astype(np.float32)
    ((y_hat * dev(gy)).sum() + (y_comp * dev(gc)).sum()).backward()
    assert np.abs(host(fake.nn_out.grad) - g["g_nn_out"]).max() <= 1e-6
    m_new, x_new, per = ops.hole_update(dev(1 - v_t), dev(v_map)[:, :, 0], y_comp.detach()[:, :, 0])
    assert np.array_equal(host(m_new), g["m_new"])
    assert np.array_equal(host(x_new), g["x_new"])
    assert float(per) == pytest.approx(float(g["inp_per"]), rel=1e-5)
    assert np.array_equal(host(mtb.trivial_copy(dev(x_t), dev(x_al), dev(v_map))), g["trivial"])
    # strided (frame-major) inputs, as produced by the warp kernel
    xa_fm = dev(x_al).transpose(1, 2).contiguous().transpose(1, 2)
    assert np.array_equal(host(ops.chn_pack(dev(x_t), dev(v_t), xa_fm, dev(v_al), dev(v_map))),
                          g["nn_input"])


@pytest.mark.parametrize("name", sorted(cases.CHNLOSS_CASES))
def test_chn_l1_terms(mtb, name):
    """One-pass L1 terms of CHN.compute_loss against the reference's golden outputs, the oracle, the
    three separate masked_l1 launches, and through the patched CHN.compute_loss."""
    import sys
    import types
    from master_thesis_b200 import ops
    y_target, v_target, y_hat, y_comp, v_map = cases.chnloss_inputs(cases.CHNLOSS_CASES[name])
    g = load_golden("chnloss_" + name)
    yh, yc = dev(y_hat).requires_grad_(True), dev(y_comp).requires_grad_(True)
    l_nh, l_vh, l_nvh = ops.chn_l1_terms(dev(y_target), dev(v_target), yh, yc, dev(v_map))
    (l_nh + l_vh + l_nvh).backward()
    got = np.array([float(l_nh), float(l_vh), float(l_nvh)], np.float32)
    assert np.allclose(got, g["losses"], rtol=1e-5, atol=0)
    ol, og_yh, og_yc = oracle.chn_l1_terms(y_target, v_target, y_hat, y_comp, v_map, grads=True)
    assert np.allclose(got, ol, rtol=1e-5, atol=0)
    for t, ref, orc in ((yh.grad, g["g_y_hat"], og_yh), (yc.grad, g["g_y_hat_comp"], og_yc)):
        scale = max(1e-12, np.abs(ref).max())
        assert np.abs(host(t) - ref).max() <= 1e-6 * scale and np.abs(host(t) - orc).max() <= 1e-6 * scale
    # the three separate launches (LossesUtils.masked_l1 mirror) give the same numbers
    f = y_hat.shape[2]
    tgt = dev(y_target).unsqueeze(2).expand(-1, -1, f, -1, -1)
    nh = dev(v_target).unsqueeze(2).expand(-1, -1, f, -1, -1)
    sep = [mtb.LossesUtils.masked_l1(dev(y_hat), tgt, nh, reduction='sum', weight=0.5),
           mtb.LossesUtils.masked_l1(dev(y_hat), tgt, dev(v_map), reduction='sum', weight=2),
           mtb.LossesUtils.masked_l1(dev(y_comp), tgt, (1 - nh) - dev(v_map), reduction='sum', weight=1)]
    assert np.allclose(got, [float(x) for x in sep], rtol=1e-6, atol=0)
    # through the plug point: CHN.compute_loss with the reference's other two terms stubbed
    stub = types.ModuleType("master_thesis")

    class _LU(object):
        perceptual = staticmethod(lambda *a, **k: (torch.zeros((), device="cuda"), None, None))
        grad = staticmethod(lambda *a, **k: torch.zeros((), device="cuda"))

    stub.LossesUtils = _LU
    saved = sys.modules.get("master_thesis")
    sys.modules["master_thesis"] = stub
    try:
        fake = types.SimpleNamespace(model_vgg=None)
        loss, items = mtb.plug.chn_compute_loss(fake, dev(y_target), dev(v_target), dev(y_hat), dev(y_comp),
                                                dev(v_map))
    finally:
        if saved is None:
            del sys.modules["master_thesis"]
        else:
            sys.modules["master_thesis"] = saved
    assert len(items) == 5 and float(loss) == pytest.approx(float(g["losses"].sum()), rel=1e-5)


def test_inference_step_fusions(mtb):
    """SURVEY 8f-2: warp + CNN-input pack in one kernel and composite + hole update in one kernel are
    bit-identical to the four-kernel route, to the golden vectors of the reference, and are what the
    inpainting loop's step uses when the aligner is a patched DFPN / CPN."""
    from master_thesis_b200 import ops, plug
    # (1) warp + pack == pack(warp), dense flow (DFPN) and theta (CPN)
    x, m, m_t, flow = cases.warp_inputs(cases.WARP_CASES["f1_odd"])
    _, _, theta = cases.cpn_inputs(cases.CPN_CASES["rand_f4"])[1:]
    r = cases.synth.rng(5)
    x_t = r.random_sample((x.shape[0], 3) + x.shape[-2:]).astype(np.float32)
    for grid, flags, xx, mm, mt_ in (
            (flow, ops.ALIGN_CORNERS | ops.VIS_FROM_MASK, x, m, m_t),
            (theta, ops.GRID_AFFINE | ops.VIS_BILINEAR | ops.VIS_FROM_MASK) + cases.cpn_inputs(cases.CPN_CASES["rand_f4"])[:3]):
        xt = dev(r.random_sample((xx.shape[0], 3) + xx.shape[-2:]).astype(np.float32))
        vt = 1 - dev(mt_)
        xa, va, vm = ops.warp_fwd(dev(xx), dev(mm), dev(grid), dev(mt_), flags)
        want = ops.chn_pack(xt, vt, xa, va, vm)
        nn_in, vm2, xa2, va2 = ops.warp_pack_fwd(dev(xx), dev(mm), dev(grid), dev(mt_), xt, vt, flags, want_aligned=True)
        assert torch.equal(nn_in, want) and torch.equal(vm2, vm) and torch.equal(xa2, xa) and torch.equal(va2, va)
        nn_in3, vm3, xa3, va3 = ops.warp_pack_fwd(dev(xx), dev(mm), dev(grid), dev(mt_), xt, vt, flags)
        assert torch.equal(nn_in3, want) and torch.equal(vm3, vm) and xa3 is None and va3 is None
    # (2) composite + hole update == the two kernels == golden (F = 1 case of the reference run)
    x_t, v_t, x_al, v_al, v_map, nn_out = cases.chn_inputs(cases.CHN_CASES["f1_odd"])
    g = load_golden("chn_f1_odd")
    b = x_t.shape[0]
    yc, m_new, x_new, per = ops.chn_fill(dev(nn_out), dev(x_t), dev(v_t), dev(1 - v_t), dev(v_map)[:, :, 0])
    assert np.array_equal(host(yc), g["y_hat_comp"][:, :, 0]) and np.array_equal(host(m_new), g["m_new"])
    assert np.array_equal(host(x_new), g["x_new"]) and float(per) == pytest.approx(float(g["inp_per"]), rel=1e-5)
    # (3) the inpainting step: fused route (patched aligner class) == generic route (foreign aligner)
    x, m, m_t, flow = cases.warp_inputs(cases.WARP_CASES["f1_odd"])
    nn_o = dev(cases.synth.nn_output(9, x.shape[0], x.shape[-2], x.shape[-1]))

    class _DFPNLike(object):
        align = plug.dfpn_align

        def __call__(self, *a):
            return None, None, None, dev(flow)

    class _Foreign(object):
        def align(self, x_target, m_target, x_refs, m_refs):
            return plug.dfpn_align_tail(x_refs, m_refs, m_target, dev(flow))

    class _CHNLike(object):
        forward = plug.chn_forward

        def nn(self, inp):
            return nn_o

        def __call__(self, *a):
            return self.forward(*a)

    xt = dev(r.random_sample((x.shape[0], 3) + x.shape[-2:]).astype(np.float32))
    fused = plug._fill_step(_CHNLike(), _DFPNLike(), xt, dev(m_t), dev(x), dev(m))
    plain = plug._fill_step(_CHNLike(), _Foreign(), xt, dev(m_t), dev(x), dev(m))
    for a_, b_ in zip(fused, plain):
        assert torch.equal(a_, b_)


def _inpaint_harness(spec, x, m, flows, nn_outs, fused, sync_every=1, by_content=False):
    """Stand-ins for the CHN module and its DFPN aligner around the patched loops: the DFPN forward and the
    RRDBNet hand out preset tensors - in call order (as make_golden.py's stand-ins do), or chosen by the content
    of their inputs (``by_content``: a step that is repeated on the same state gets the same tensors)."""
    from master_thesis_b200 import plug

    def pick(presets, counter, t):
        if by_content:
            return dev(presets[int(float(t.double().abs().sum()) * 1000.0) % len(presets)])
        return dev(presets[counter % len(presets)])

    class _DFPNLike(object):
        def __init__(self):
            self.n = 0

        def __call__(self, x_target, m_target, x_refs, m_refs):
            self.n += 1
            return None, None, None, pick(flows, self.n - 1, m_target + x_refs[:, :1, 0])

    if fused:
        _DFPNLike.align = plug.dfpn_align
    else:
        _DFPNLike.align = lambda self, xt, mt_, xr, mr: plug.dfpn_align_tail(xr, mr, mt_, self(xt, mt_, xr, mr)[3])

    class _CHNLike(object):
        forward = plug.chn_forward
        inpaint_ff = plug.chn_inpaint_ff
        inpaint_ip = plug.chn_inpaint_ip
        get_indexes_ff = staticmethod(cases.get_indexes_ff)
        get_indexes_ip = staticmethod(cases.get_indexes_ip)
        mt_b200_sync_every = sync_every

        def __init__(self):
            self.model_aligner = _DFPNLike()
            self.k = 0

        def nn(self, inp):
            self.k += 1
            return pick(nn_outs, self.k - 1, inp[:, 6:])      # the three visibility channels of the CNN input

        def __call__(self, *a):
            return self.forward(*a)

    chn = _CHNLike()
    algo = chn.inpaint_ip if spec.get("algo") == "ip" else chn.inpaint_ff
    y = algo(dev(x).clone(), dev(m).clone(), s=1, D=20, e=spec.get("e", 1))
    return host(y), chn.k


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("name", sorted(cases.INPAINT_CASES))
def test_inpaint_mirrors(mtb, name, fused):
    """The patched CHN.inpaint_ff / inpaint_ip (two fused kernels per step, or the four-kernel route a foreign
    aligner takes) against the output of the unmodified reference loops, bit for bit."""
    spec = cases.INPAINT_CASES[name]
    x, m, flows, nn_outs = cases.inpaint_inputs(spec)
    g = load_golden("inpaint_" + name)
    y, k = _inpaint_harness(spec, x, m, flows, nn_outs, fused)
    assert k == int(g["steps"][0])
    assert np.array_equal(y, g["y"])


@pytest.mark.parametrize("sync_every", [2, 3, 8])
@pytest.mark.parametrize("name", sorted(cases.INPAINT_CASES))
def test_inpaint_device_side_loop_control(mtb, name, sync_every):
    """SURVEY 8f-4: with the loop condition evaluated on the device (gated fill step) and the host looking only
    every k steps, the inpainted frames are bit-identical to the one-sync-per-step loop; the surplus steps (at
    most k - 1 per target frame) run as no-ops."""
    spec = cases.INPAINT_CASES[name]
    x, m, flows, nn_outs = cases.inpaint_inputs(spec)
    y1, k1 = _inpaint_harness(spec, x, m, flows, nn_outs, True, 1, by_content=True)
    yk, kk = _inpaint_harness(spec, x, m, flows, nn_outs, True, sync_every, by_content=True)
    assert np.array_equal(yk, y1)
    assert k1 <= kk <= k1 + (sync_every - 1) * x.shape[1]
    assert k1 > x.shape[1] or "long" not in name      # the long cases really iterate


def test_no_out_of_bounds_writes(mtb):
    """Every output and workspace the ops allocate is carved out of a larger sentinel-filled buffer; after
    the calls the guard bands before and after each allocation must be untouched (compute-sanitizer is not
    available on this pool).  Shapes are ragged on purpose: partial tiles, partial 1024-pixel chunks,
    channel counts that are not multiples of the slabs, widths that are not multiples of 4."""
    import contextlib
    from master_thesis_b200 import _lib, ops, plug
    G = 256  # guard elements on both sides (keeps 16 B alignment for every dtype)
    made = []

    def guarded_empty(*a, **k):
        probe = torch.empty(*a, **{**k, "device": "meta"})
        n = probe.numel()
        buf = torch.empty(n + 2 * G, dtype=probe.dtype, device=k.get("device", "cuda"))
        sentinel = 0xA5 if probe.dtype == torch.uint8 else -12345.0
        buf.fill_(sentinel)
        made.append((buf, n, sentinel))
        return _lib.keep(buf[G:G + n].view(probe.shape))

    @contextlib.contextmanager
    def guards():
        orig, orig_like = ops._empty, ops._empty_like
        saved_ws = dict(ops._workspaces)
        ops._workspaces.clear()
        ops._empty = guarded_empty
        ops._empty_like = lambda t, **k: guarded_empty(t.shape, dtype=t.dtype, device=t.device)
        try:
            yield
        finally:
            ops._empty, ops._empty_like = orig, orig_like
            ops._workspaces.clear()
            ops._workspaces.update(saved_ws)

    r = cases.synth.rng(123)
    with guards():
        # staged CPN warp with partial tiles, direct-gather warp with W % 4 != 0
        x, m, m_t, theta = cases.cpn_inputs(STAGED_CASES["rand"])
        mtb.cpn_align_tail(dev(x), dev(m), dev(m_t), dev(theta))
        xw, mw, mtw, flow = cases.warp_inputs(cases.WARP_CASES["f1_odd"])
        mtb.dfpn_align_tail(dev(xw), dev(mw), dev(mtw), dev(flow))
        # warp + pack, composite + hole update (odd sizes)
        xt = dev(r.random_sample((xw.shape[0], 3) + xw.shape[-2:]).astype(np.float32))
        nn_in, vm, _, _ = ops.warp_pack_fwd(dev(xw), dev(mw), dev(flow), dev(mtw), xt, 1 - dev(mtw),
                                            ops.ALIGN_CORNERS | ops.VIS_FROM_MASK, want_aligned=True)
        nn_o = dev(cases.synth.nn_output(9, xw.shape[0], xw.shape[-2], xw.shape[-1]))
        ops.chn_fill(nn_o, xt, 1 - dev(mtw), dev(mtw), vm[:, :, 0])
        # CHN pack / composite / the three L1 terms forward + backward
        x_t, v_t, x_al, v_al, v_map, nn_out = cases.chn_inputs(cases.CHN_CASES["f1_odd"])
        ops.chn_pack(dev(x_t), dev(v_t), dev(x_al), dev(v_al), dev(v_map))
        no = dev(nn_out).requires_grad_(True)
        yh, yc = ops.chn_composite(no, dev(x_t), dev(v_t), x_t.shape[0], x_al.shape[2])
        y_target, v_target, y_hat, y_comp, v_map2 = cases.chnloss_inputs(cases.CHNLOSS_CASES["f1_odd"])
        yh2, yc2 = dev(y_hat).requires_grad_(True), dev(y_comp).requires_grad_(True)
        sum(ops.chn_l1_terms(dev(y_target), dev(v_target), yh2, yc2, dev(v_map2))).backward()
        # CM: both weight paths, ragged shapes
        for shape in ((5, 4, 9, 24, 48), (3, 2, 5, 32, 32)):
            b, f, c, h, w = shape
            cf, vt, va = cases.synth.cm_inputs(61 + b, b, f, c, h, w, 4)
            for table in (2, 1, 0):
                try:
                    _set_tuning("MT_CM_TABLE", table)
                    ops.cm_match(dev(cf), dev(vt), dev(va))
                finally:
                    _set_tuning("MT_CM_TABLE", 2)
        # correlation and the fused DFPN loss
        ft, vtt, fr, vr = cases.synth.vgg_feats(5, 1, 2)
        ops.corr4d(dev(ft), dev(vtt), dev(fr), dev(vr))
        torch.cuda.synchronize()
    assert len(made) > 30
    for buf, n, sentinel in made:
        lo, hi = buf[:G], buf[G + n:]
        assert bool((lo == sentinel).all()) and bool((hi == sentinel).all()), "guard band overwritten (n=%d)" % n


# ---------------------------------------------------------------- full-size properties
def test_full_size_properties(mtb):
    """BASELINE cfg2 sizes (B=8, F=4, 256x256): size-independent properties."""
    from master_thesis_b200 import ops, synth
    b, f, h, w = 8, 4, 256, 256
    x, m, _ = synth.frames(7, b, f + 1, h, w)
    xr, mr, mt_ = dev(x[:, :, 1:]), dev(m[:, :, 1:]), dev(m[:, :, 0])
    # (1) identity flow: the warp is the identity (to fp32 noise of the grid itself), the
    #     nearest visibility is exact, and v_map = clamp(v_al - (1 - m_t))
    ident = dev(np.broadcast_to(synth.identity_grid(h, w, True), (b, f, h, w, 2)).copy())
    xa, va, vm = mtb.dfpn_align_tail(xr, mr, mt_, ident)
    assert (xa - xr).abs().max() <= 1e-4 and torch.equal(va, 1 - mr)   # 1 ulp of the grid = 1.5e-5 px
    assert torch.equal(vm, (va - (1 - mt_).unsqueeze(2)).clamp(0, 1))
    # (2) integer translation by (dx, dy) pixels == shifted frame with zero padding
    dx, dy = 5, -3
    shift = ident.clone()
    shift[..., 0] += 2.0 * dx / (w - 1)
    shift[..., 1] += 2.0 * dy / (h - 1)
    xa, va, _ = mtb.dfpn_align_tail(xr, mr, mt_, shift)
    ref = torch.zeros_like(xr)
    ref[..., 3:, :w - dx] = xr[..., :h - 3, dx:]
    inner = (slice(None),) * 3 + (slice(8, h - 8), slice(8, w - 8))
    assert (xa[inner] - ref[inner]).abs().max() <= 1e-4
    # (3) affine identity theta == dense identity grid path (align_corners=False)
    theta = dev(synth.thetas(0, b * f, 0.0))
    xa, va, vm = mtb.cpn_align_tail(xr, mr, mt_, theta)
    assert (xa - xr).abs().max() <= 1e-4 and torch.equal(va, 1 - mr)   # 1 ulp of the grid = 1.5e-5 px
    # (4) oracle spot check on one sample at full resolution
    flow = synth.dense_flow(9, 1, f, h, w, 0.05, True)
    xa, va, vm = mtb.dfpn_align_tail(xr[:1], mr[:1], mt_[:1], dev(flow))
    oxa, ova, ovm = oracle.dfpn_align_tail(x[:1, :, 1:], m[:1, :, 1:], m[:1, :, 0], flow)
    assert np.array_equal(host(xa), oxa) and np.array_equal(host(va), ova) and np.array_equal(host(vm), ovm)
    # (5) CM at full size: scaling c_feats of one reference by 0 removes it (weights renormalise)
    cf, vt, vaa = synth.cm_inputs(3, 2, 5, 128, 64, 64)
    out, cmask = ops.cm_match(dev(cf), dev(vt), dev(vaa))
    oout, ocm = oracle.cm_module(cf, vt, vaa)
    assert np.abs(host(out) - oout).max() <= 1e-5 and np.abs(host(cmask) - ocm).max() <= 2e-6
    # (6) correlation at the real shape: cosine bounds, symmetry of self-correlation
    ft, vt_, fr, vr = synth.vgg_feats(5, 2, 2)
    c = ops.corr4d(dev(ft), None, dev(ft).unsqueeze(2), None)
    assert float(c.max()) <= 1.0 + 1e-2 and float(c.min()) >= -1e-3
    c2 = c[:, 0].reshape(2, 256, 256)
    assert (c2 - c2.transpose(1, 2)).abs().max() <= 2e-3
    assert (torch.diagonal(c2, dim1=1, dim2=2) - 1).abs().max() <= 2e-3


def test_480x854_davis_shape(mtb):
    """cfg4 shape: non-square, W % 4 != 0 (plane still 16 B aligned)."""
    from master_thesis_b200 import synth
    b, f, h, w = 1, 1, 480, 854
    x, m, _ = synth.frames(17, b, f + 1, h, w)
    flow = synth.dense_flow(18, b, f, h, w, 0.03, True)
    xa, va, vm = mtb.dfpn_align_tail(dev(x[:, :, 1:]), dev(m[:, :, 1:]), dev(m[:, :, 0]), dev(flow))
    oxa, ova, ovm = oracle.dfpn_align_tail(x[:, :, 1:], m[:, :, 1:], m[:, :, 0], flow)
    assert np.array_equal(host(xa), oxa) and np.array_equal(host(va), ova) and np.array_equal(host(vm), ovm)


# ---------------------------------------------------------------- host-buffer C ABI
def test_host_buffer_entry_points(mtb):
    """mt_cpn_align_host / mt_dfpn_align_host: plain host pointers in, host pointers out (H2D, kernel, D2H and
    the synchronisation inside the call) - what a non-torch caller of the C ABI uses."""
    import ctypes
    from master_thesis_b200 import _lib
    lib = _lib.load()
    p = lambda a: ctypes.c_void_p(a.ctypes.data)   # noqa: E731
    for spec, staged in ((cases.CPN_CASES["rand_f4"], False), (STAGED_CASES["rand"], True)):
        x, m, m_t, theta = cases.cpn_inputs(spec)
        b, _, f, h, w = x.shape
        xa, va, vm = np.full_like(x, -7.0), np.full_like(m, -7.0), np.full_like(m, -7.0)
        rc = lib.mt_cpn_align_host(p(x), p(m), p(m_t), p(theta), p(xa), p(va), p(vm), b, f, h, w)
        assert rc == 0, _lib.last_error()
        oxa, ova, ovm = oracle.cpn_align_tail(x, m, m_t, theta=theta)
        assert np.array_equal(xa, oxa) and np.array_equal(va, ova) and np.array_equal(vm, ovm)
    for name in ("smooth_f4", "noisy_oob", "f1_odd"):
        x, m, m_t, flow = cases.warp_inputs(cases.WARP_CASES[name])
        g = load_golden("warp_" + name)
        b, _, f, h, w = x.shape
        xa, va, vm = np.full_like(x, -7.0), np.full_like(m, -7.0), np.full_like(m, -7.0)
        rc = lib.mt_dfpn_align_host(p(x), p(m), p(m_t), p(flow), p(xa), p(va), p(vm), b, f, h, w)
        assert rc == 0, _lib.last_error()
        assert np.array_equal(xa, g["x_aligned"]) and np.array_equal(va, g["v_aligned"]) and np.array_equal(vm, g["v_map"])
    # errors are codes + messages, never exceptions or crashes
    assert lib.mt_dfpn_align_host(None, p(m), p(m_t), p(flow), p(xa), p(va), p(vm), b, f, h, w) == -1
    assert "NULL" in _lib.last_error()
    assert lib.mt_cpn_align_host(p(x), p(m), p(m_t), p(flow), p(xa), p(va), p(vm), 0, f, h, w) == -1


# ---------------------------------------------------------------- reductions at the full batch sizes
def test_fused_losses_at_cfg3_and_cfg5_sizes(mtb):
    """warp_l1_fwd / bwd at the cfg3 batch (B=32, F=4, 256 x 256: 8.4 M pixels x 3 channels through the
    per-CTA partials + last-CTA double sum) and chn_l1x3 at the same pixel count, against the CPU oracle."""
    from master_thesis_b200 import ops, synth
    b, f, h, w = 32, 4, 256, 256
    x, m, _ = synth.frames(201, b, f + 1, h, w)
    xr, vr = np.ascontiguousarray(x[:, :, 1:]), np.ascontiguousarray(1 - m[:, :, 1:])
    xt, vt = np.ascontiguousarray(x[:, :, 0]), np.ascontiguousarray(1 - m[:, :, 0])
    flow = synth.dense_flow(202, b, f, h, w, 0.3, True)          # a few percent of the samples out of frame
    fl = dev(flow).requires_grad_(True)
    loss = mtb.LossesUtils.alignment_recons(dev(xt), dev(vt), dev(xr), dev(vr), fl)
    loss.backward()
    oxa, _ = oracle.align_set(xr, vr, flow)
    y_hat = np.repeat(xt[:, :, None], f, axis=2)
    mask = np.repeat(vt[:, :, None], f, axis=2) * (1 - oracle.mask_out(flow))
    oloss = oracle.masked_l1(y_hat, oxa, mask, reduction="sum")
    assert float(loss) == pytest.approx(oloss, rel=1e-5)
    og = oracle.align_set_bwd_flow(xr, flow, oracle.masked_l1_bwd(y_hat, oxa, mask, reduction="sum"))
    assert np.abs(host(fl.grad) - og).max() <= 2e-5 * np.abs(og).max()
    del oxa, y_hat, mask, og, fl
    # the three L1 terms of CHN.compute_loss at the same size
    r = synth.rng(203)
    y_target = r.random_sample((b, 3, h, w)).astype(np.float32)
    v_target = (r.random_sample((b, 1, h, w)) < 0.85).astype(np.float32)
    y_hat = r.random_sample((b, 3, f, h, w)).astype(np.float32)
    v_al = (r.random_sample((b, 1, f, h, w)) < 0.8).astype(np.float32)
    v_map = np.clip(v_al - v_target[:, :, None], 0, 1).astype(np.float32)
    y_comp = (v_target[:, :, None] * y_target[:, :, None] + (1 - v_target[:, :, None]) * y_hat).astype(np.float32)
    yh, yc = dev(y_hat).requires_grad_(True), dev(y_comp).requires_grad_(True)
    terms = ops.chn_l1_terms(dev(y_target), dev(v_target), yh, yc, dev(v_map))
    sum(terms).backward()
    ol, og_yh, og_yc = oracle.chn_l1_terms(y_target, v_target, y_hat, y_comp, v_map, grads=True)
    assert np.allclose([float(t) for t in terms], ol, rtol=1e-5, atol=0)
    assert np.abs(host(yh.grad) - og_yh).max() <= 1e-6 * np.abs(og_yh).max()
    assert np.abs(host(yc.grad) - og_yc).max() <= 1e-6 * max(1e-12, np.abs(og_yc).max())


# ---------------------------------------------------------------- ADVICE r1
def test_masked_l1_broadcast_masks(mtb):
    """masked_l1 with masks smaller than y_hat (the shapes utils.py:139-157 documents): the 'sum' denominator is
    torch.sum(mask) of the mask as given.  Forward and backward against the unmodified reference's outputs."""
    y4a, y4b, m4, y5a, y5b, m5f, m5b, m5p = cases.l1_broadcast_inputs()
    g = load_golden("l1_broadcast")
    for key, (ya, yb, mk) in dict(l4=(y4a, y4b, m4), l5f=(y5a, y5b, m5f), l5b=(y5a, y5b, m5b),
                                  l5p=(y5a, y5b, m5p)).items():
        a = dev(ya).requires_grad_(True)
        loss = mtb.LossesUtils.masked_l1(a, dev(yb), dev(mk), reduction='sum', weight=1.5)
        loss.backward()
        assert float(loss) == pytest.approx(float(g[key]), rel=1e-5), key
        assert np.abs(host(a.grad) - g["g_" + key]).max() <= 1e-6 * np.abs(g["g_" + key]).max(), key
        mean = mtb.LossesUtils.masked_l1(dev(ya), dev(yb), dev(mk), reduction='mean')
        assert float(mean) == pytest.approx(float(g[key + "_mean"]), rel=1e-5), key
    # mask=None is torch.ones_like(y_hat) (the flow losses of DFPN.compute_loss) without the tensor
    from master_thesis_b200 import ops
    ones = ops.masked_l1(dev(y5a), dev(y5b), torch.ones_like(dev(y5a)), reduction='sum')
    none = ops.masked_l1(dev(y5a), dev(y5b), None, reduction='sum')
    assert float(ones) == pytest.approx(float(none), rel=1e-6)


def test_warp_pack_without_v_map_output(mtb):
    """mt_warp_pack_fwd with v_map = NULL (allowed by the header): channel 8 of nn_in is still the v_map."""
    from master_thesis_b200 import ops
    x, m, m_t, flow = cases.warp_inputs(cases.WARP_CASES["f1_odd"])
    r = cases.synth.rng(6)
    xt = dev(r.random_sample((x.shape[0], 3) + x.shape[-2:]).astype(np.float32))
    flags = ops.ALIGN_CORNERS | ops.VIS_FROM_MASK
    want, vm, _, _ = ops.warp_pack_fwd(dev(x), dev(m), dev(flow), dev(m_t), xt, 1 - dev(m_t), flags)
    got, none, _, _ = ops.warp_pack_fwd(dev(x), dev(m), dev(flow), dev(m_t), xt, 1 - dev(m_t), flags, want_v_map=False)
    assert none is None and torch.equal(got, want) and torch.equal(got[:, 8], vm[:, 0].reshape(got[:, 8].shape))


def test_staged_warp_with_expanded_inputs(mtb):
    """Stride-0 (expanded) inputs cannot be encoded in a tensor map: the CPN tail must take the direct kernel
    and still match the oracle (one target mask / one reference clip shared by the whole batch)."""
    spec = STAGED_CASES["rand"]
    x, m, m_t, theta = cases.cpn_inputs(spec)
    b = x.shape[0]
    m_t1 = np.ascontiguousarray(m_t[:1])
    xa, va, vm = mtb.cpn_align_tail(dev(x), dev(m), dev(m_t1).expand(b, -1, -1, -1), dev(theta))
    oxa, ova, ovm = oracle.cpn_align_tail(x, m, np.repeat(m_t1, b, axis=0), theta=theta)
    assert np.array_equal(host(xa), oxa) and np.array_equal(host(va), ova) and np.array_equal(host(vm), ovm)
    x1, m1 = np.ascontiguousarray(x[:1]), np.ascontiguousarray(m[:1])
    xa, va, vm = mtb.cpn_align_tail(dev(x1).expand(b, -1, -1, -1, -1), dev(m1).expand(b, -1, -1, -1, -1), dev(m_t), dev(theta))
    oxa, ova, ovm = oracle.cpn_align_tail(np.repeat(x1, b, axis=0), np.repeat(m1, b, axis=0), m_t, theta=theta)
    assert np.array_equal(host(xa), oxa) and np.array_equal(host(va), ova) and np.array_equal(host(vm), ovm)


def test_operators_without_backward_refuse_differentiable_inputs(mtb):
    from master_thesis_b200 import ops
    cf, vt, va = cases.cm_inputs(cases.CM_CASES["small"])
    with pytest.raises(RuntimeError, match="no backward"):
        ops.cm_match(dev(cf).requires_grad_(True), dev(vt), dev(va))
    ft, vt_, fr, vr = cases.corr_inputs(cases.CORR_CASES["small_masked"])
    with pytest.raises(RuntimeError, match="no backward"):
        ops.corr4d(dev(ft).requires_grad_(True), dev(vt_), dev(fr), dev(vr))
    x, m, m_t, flow = cases.warp_inputs(cases.WARP_CASES["f1_odd"])
    with pytest.raises(RuntimeError, match="no backward"):
        mtb.dfpn_align_tail(dev(x), dev(m), dev(m_t), dev(flow).requires_grad_(True))
    with torch.no_grad():      # the reference's own flows (frozen aligner, no_grad) are unaffected
        mtb.dfpn_align_tail(dev(x), dev(m), dev(m_t), dev(flow).requires_grad_(True))


# ---------------------------------------------------------------- f1: flow resize fused into the warp
@pytest.mark.parametrize("name", sorted(cases.LOWRES_CASES))
def test_lowres_flow_align(mtb, name):
    """The DFPN.align tail fed with the 256 x 256 flow: resize_flow (model_dfpn.py:100-101) happens inside the
    warp kernel; bit-identical to the unmodified reference (resize, then align) and to the two-step route."""
    from master_thesis_b200 import ops, plug
    x, m, m_t, flow256 = cases.lowres_inputs(cases.LOWRES_CASES[name])
    g = load_golden("lowres_" + name)
    xa, va, vm = mtb.dfpn_align_tail(dev(x), dev(m), dev(m_t), dev(flow256))
    cases.lowres_check(host(xa), host(va), host(vm), g)
    flow_hw = oracle.resize_flow(flow256, x.shape[-2:])
    xa2, va2, vm2 = mtb.dfpn_align_tail(dev(x), dev(m), dev(m_t), dev(flow_hw))
    assert torch.equal(xa, xa2) and torch.equal(va, va2) and torch.equal(vm, vm2)
    # warp + CNN-input pack with the low-resolution flow == pack(warp)
    r = cases.synth.rng(8)
    xt = dev(r.random_sample((x.shape[0], 3) + x.shape[-2:]).astype(np.float32))
    flags = ops.ALIGN_CORNERS | ops.VIS_FROM_MASK
    nn_in, vm3, xa3, va3 = ops.warp_pack_fwd(dev(x), dev(m), dev(flow256), dev(m_t), xt, 1 - dev(m_t), flags, want_aligned=True)
    assert torch.equal(nn_in, ops.chn_pack(xt, 1 - dev(m_t), xa, va, vm)) and torch.equal(vm3, vm) and torch.equal(xa3, xa)

    # through the aligner protocol: a patched DFPN hands the kernel its 256 x 256 flow
    class _DFPNLike(object):
        align = plug.dfpn_align

        def _mt_b200_flow_256(self, *a):
            return dev(flow256)

        def __call__(self, *a):
            raise AssertionError("the full-resolution forward must not be used for frames that are not 256 x 256")

    xa4, va4, vm4 = _DFPNLike().align(dev(x[:, :, 0]), dev(m_t), dev(x), dev(m))
    assert torch.equal(xa4, xa) and torch.equal(vm4, vm)


# ---------------------------------------------------------------- a1 + a4 + a5 + a6 in context
def _stub_reference_package():
    """A stand-in ``master_thesis`` package for the GPU box (the reference is absent there): the two helpers the
    DFPN mirrors look up on it, restated in oracle/torch_port.py (pinned to the reference on the CPU)."""
    import types
    from oracle import torch_port as tp
    stub = types.ModuleType("master_thesis")
    stub.TransformsUtils = types.SimpleNamespace(resize_set=tp.resize_set)
    stub.FlowsUtils = types.SimpleNamespace(resize_flow=tp.resize_flow)
    return stub


@pytest.mark.parametrize("name", sorted(cases.DFPNLOSS_CASES))
def test_dfpn_training_step_mirrors(mtb, name):
    """The patched DFPN._train_val_wrapper + DFPN.compute_loss (fused warp + mask_out + masked-L1 kernels, no
    aligned frames in HBM) against the golden outputs of the unmodified reference methods: loss items, and
    the gradients that reach the flows and the correlation volume."""
    import sys
    from master_thesis_b200 import _lib, plug
    spec = cases.DFPNLOSS_CASES[name]
    x, m, y, flow_gt, use, corr, f16, f64, fhw, feats = cases.dfpnloss_inputs(spec)
    g = load_golden("dfpnloss_" + name)
    n = x.shape[2]
    t, r_list = n // 2, [i for i in range(n) if i != n // 2]
    leaves = [dev(a).requires_grad_(True) for a in (corr, f16, f64, fhw)]

    class _DFPNLike(object):
        def __call__(self, *a):
            return tuple(leaves)

        def model_vgg(self, inp):
            return [None, None, None, dev(feats)]

    saved = sys.modules.get("master_thesis")
    sys.modules["master_thesis"] = _stub_reference_package()
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
    assert len(res) == 8 and all(isinstance(a, plug.DeferredAlign) for a in res[4])
    # the hot path of the step is exactly these launches: no align_set, no mask_out, no x_aligned in HBM
    assert sorted(plan.names()) == sorted(["mt_corr4d_vgg_l1_fwd", "mt_corr4d_l1_bwd"] + ["mt_masked_l1_fwd"] * 3 +
                                          ["mt_warp_l1_fwd"] * 2 + ["mt_warp_l1_bwd"] * 2 + ["mt_masked_l1_bwd"] * 3)
    # corr_loss compares a TF32 correlation of the ground truth with the given volume: |d| <= 7e-4 per element
    assert abs(float(items[0]) - float(g["items"][0])) <= 1e-3
    assert float(loss) - float(items[0]) == pytest.approx(float(g["loss"]) - float(g["items"][0]), rel=1e-5)
    assert np.allclose([float(i) for i in items[1:]], g["items"][1:], rtol=1e-5, atol=0)
    assert np.abs(host(grads[2]) - g["g_flow64"]).max() <= 2e-5 * np.abs(g["g_flow64"]).max()
    assert np.abs(host(grads[3]) - g["g_flowhw"]).max() <= 2e-5 * np.abs(g["g_flowhw"]).max()
    assert float(grads[1].abs().double().sum()) == pytest.approx(float(g["g_flow16_abs"]), rel=1e-5)
    assert float(grads[0].abs().double().sum()) == pytest.approx(float(g["g_corr_abs"]), rel=1e-3)
    # a consumer that treats an xs_aligned entry as a tensor gets the aligned frames
    assert float(res[4][2].double().sum()) == pytest.approx(float(g["xhw_al_sum"]), rel=1e-6)
    assert float(torch.sum(res[4][1]).double()) == pytest.approx(float(g["x64_al_sum"]), rel=1e-5)


# ---------------------------------------------------------------- f3: CorrelationVGG.forward neighbours
@pytest.mark.parametrize("tn", [0, 64, 128, 256])
@pytest.mark.parametrize("name", sorted(cases.CORRVGG_CASES))
def test_corr_vgg_forward_mirror(mtb, name, tn):
    """The patched CorrelationVGG.forward: strided (un-permuted) VGG features and full-resolution masks go
    straight into the tensor-core kernel; against the unmodified reference's output and the CPU oracle."""
    from master_thesis_b200 import _lib, plug
    spec = cases.CORRVGG_CASES[name]
    x_t, m_t, x_r, m_r, ft, fr = cases.corrvgg_inputs(spec)
    g = load_golden("corrvgg_" + name)
    b, f = spec["b"], spec["f"]

    class _CorrLike(object):
        use_softmax = False
        conv = staticmethod(lambda c: c)

        def __init__(self):
            self.n = 0

        def model_vgg(self, inp, normalize_input=True):
            self.n += 1
            return [None, None, None, dev(ft) if self.n == 1 else dev(fr)]

    try:
        _set_tuning("MT_CORR_TN", tn)
        with _lib.record() as plan:
            c = host(plug.corr_vgg_forward(_CorrLike(), dev(x_t), dev(m_t), dev(x_r), dev(m_r)))
    finally:
        _set_tuning("MT_CORR_TN", 0)
    assert plan.names() == ["mt_corr4d_vgg_fwd"]      # no permute copy, no mask kernels
    cases.corr_check(c, g, spec, 2e-3)
    feats_r = fr.reshape(b, f, 512, 16, 16).transpose(0, 2, 1, 3, 4)
    o = oracle.corr4d(ft, oracle.vis_nearest(m_t, (16, 16)), feats_r, oracle.vis_nearest(m_r, (16, 16)))
    assert np.abs(c - o).max() <= 2e-3 and np.array_equal(c == 0.0, o == 0.0)
    assert int((c.reshape(b, f, 256, 256) == 0).all(-1).sum()) == int(g["zero_rows"][0])


# ---------------------------------------------------------------- 8f-4 FlowEstimator input pack
@pytest.mark.parametrize("name", sorted(cases.FLOWPACK_CASES))
def test_flow_estimator_input_pack(mtb, name):
    """mt_flow_pack and the patched FlowEstimator.forward against the unmodified reference method
    (model_dfpn.py:714-744): CNN input, output and the gradient that reaches flow_pre, bit for bit, for every
    memory layout of flow_pre (vector paths: planar / interleaved; scalar path: odd sizes, sliced window)."""
    from master_thesis_b200 import ops, plug
    spec = cases.FLOWPACK_CASES[name]
    x_t, m_t, x_r, m_r, base, gain, up = cases.flowpack_inputs(spec)
    g = load_golden("flowpack_" + name)
    tb = dev(base).requires_grad_(True)
    flow = cases.flowpack_view(tb, spec)
    want = oracle.flow_pack(x_t, m_t, x_r, m_r, cases.flowpack_view(base, spec))
    with torch.no_grad():
        got = ops.flow_pack(dev(x_t), dev(m_t), dev(x_r), dev(m_r), flow)
    assert np.array_equal(host(got), want) and np.array_equal(host(got), g["nn_input"])
    # strided frame views (x[:, :, r_list] / x[:, :, t] of one clip tensor, as DFPN.align receives them)
    clip = dev(np.concatenate([x_t[:, :, None], x_r], axis=2))
    mclip = dev(np.concatenate([m_t[:, :, None], m_r], axis=2))
    with torch.no_grad():
        got2 = ops.flow_pack(clip[:, :, 0], mclip[:, :, 0], clip[:, :, 1:], mclip[:, :, 1:], flow)
    assert torch.equal(got2, got)
    seen = {}

    class Estimator(object):
        def nn(self, inp):
            seen["nn_input"] = inp.detach().clone()
            return inp[:, 0:2] * 0.5 + inp[:, 8:10] * dev(gain)

    out = plug.flow_estimator_forward(Estimator(), dev(x_t), dev(m_t), dev(x_r), dev(m_r), flow)
    assert tuple(out.shape) == tuple(up.shape)
    (out * dev(up)).sum().backward()
    assert np.array_equal(host(seen["nn_input"]), g["nn_input"])
    assert np.array_equal(host(out), g["flow_out"])
    assert np.array_equal(host(tb.grad), g["g_base"])


def test_flow_estimator_input_pack_full_size(mtb):
    """cfg3's 256 x 256 estimator input (32 frames here) against the oracle; the guard band past the output and
    the inputs stay untouched."""
    from master_thesis_b200 import ops, synth
    b, f, h, w = 8, 4, 256, 256
    x, m, _ = synth.frames(77, b, f + 1, h, w)
    flow = synth.dense_flow(78, b, f, h, w, 0.05, True)
    t = f // 2
    r_list = [i for i in range(f + 1) if i != t]
    xd, md = dev(x), dev(m)
    got = ops.flow_pack(xd[:, :, t], md[:, :, t], xd[:, :, r_list], md[:, :, r_list], dev(flow))
    want = oracle.flow_pack(x[:, :, t], m[:, :, t], x[:, :, r_list], m[:, :, r_list], flow)
    assert np.array_equal(host(got), want)
    assert torch.equal(xd, dev(x)) and torch.equal(md, dev(m))


# ---------------------------------------------------------------- 8f-3: F.l1_loss(corr, corr_y) in the epilogue
_CORR_L1_VARIANTS = [(0, 0, -1), (128, 64, 0), (128, 128, 0), (128, 256, 0), (256, 64, 0), (256, 128, 0),
                     (256, 256, 0), (0, 128, 1), (0, 256, 1)]


@pytest.mark.parametrize("tm,tn,pair", _CORR_L1_VARIANTS)
@pytest.mark.parametrize("name", ["real_nomask", "mid_masked", "big_masked"])
def test_corr4d_l1_in_the_epilogue(mtb, name, tm, tn, pair):
    """mt_corr4d_vgg_l1_fwd / mt_corr4d_l1_bwd (model_dfpn.py:254-257 without the ground-truth volume in HBM), every
    tile variant and the CTA-pair kernel at 2 / 40 / 128 frames: the loss against the CPU oracle (TF32 bound) and
    against the L1 of the volume the store-mode launch of the SAME variant writes (same accumulators: the signs are
    identical, the loss agrees to summation order), the gradient against autograd's formula."""
    from master_thesis_b200 import ops
    spec = cases.CORR_CASES[name]
    ft, _, fr, _ = cases.corr_inputs(spec)
    b, c, f = fr.shape[:3]
    r = np.random.RandomState(spec["seed"] + 40)
    pred = r.random_sample((b, f, 16, 16, 16, 16)).astype(np.float32)
    try:
        _set_tuning("MT_CORR_TM", tm)
        _set_tuning("MT_CORR_TN", tn)
        _set_tuning("MT_CORR_2CTA", pair)
        vol = ops.corr4d_vgg(dev(ft), None, dev(fr), None)
        p = dev(pred)
        p.view(-1)[::7] = vol.view(-1)[::7]                  # exact ties: sign 0, no gradient
        p.requires_grad_(True)
        loss = ops.corr4d_l1(p, dev(ft), dev(fr))
        (loss * 3.0).backward()
    finally:
        _set_tuning("MT_CORR_TM", 0)
        _set_tuning("MT_CORR_TN", 0)
        _set_tuning("MT_CORR_2CTA", -1)
    d = p.detach() - vol
    assert float(loss) == pytest.approx(float(d.abs().double().mean()), rel=2e-6)
    want_g = torch.sign(d) * (3.0 / d.numel())
    assert torch.allclose(p.grad, want_g, rtol=1e-6, atol=0)
    assert int((p.grad == 0).sum()) >= d.numel() // 7
    o_loss, o_grad = oracle.corr4d_l1(host(p), ft, fr)
    assert abs(float(loss) - o_loss) <= 1e-3                  # |corr_tf32 - corr_fp32| <= 2e-3 per element
    # signs differ from the fp32 oracle only where |pred - corr| is inside the TF32 error band
    flip = (host(p.grad) != 3.0 * o_grad) & (np.abs(host(d)) > 2e-3)
    assert not flip.any()


def test_corr4d_l1_strided_features_no_grad(mtb):
    """The ground-truth features as DFPN.compute_loss hands them over (the transposed view of the VGG output,
    model_dfpn.py:252) and a prediction that needs no gradient (validation): no sign tensor is written."""
    from master_thesis_b200 import ops
    spec = cases.DFPNLOSS_CASES["n5"]
    *_, corr, _, _, _, feats = cases.dfpnloss_inputs(spec)
    b, n = spec["b"], spec["n"]
    t, r_list = n // 2, [i for i in range(n) if i != n // 2]
    fy = dev(feats).reshape(b, n, -1, 16, 16).transpose(1, 2)
    with torch.no_grad():
        loss = ops.corr4d_l1(dev(corr), fy[:, :, t], fy[:, :, r_list])
    fyh = feats.reshape(b, n, -1, 16, 16).transpose(0, 2, 1, 3, 4)
    o_loss, _ = oracle.corr4d_l1(corr, fyh[:, :, t], fyh[:, :, r_list])
    assert abs(float(loss) - o_loss) <= 1e-3
    assert abs(float(loss) - float(load_golden("dfpnloss_n5")["items"][0])) <= 1e-3


def test_dfpn_align_tail_full_size(mtb):
    """cfg2-size DFPN tail (32 frames of 256 x 256, the bench's flow statistics, plus a band of flow that leaves the
    frame) and a 480 x 854 frame against the oracle, bit for bit."""
    from master_thesis_b200 import synth
    for (b, f, h, w, seed) in ((8, 4, 256, 256, 31), (1, 2, 480, 854, 32)):
        x, m, _ = synth.frames(seed, b, f + 1, h, w)
        flow = synth.dense_flow(seed + 1, b, f, h, w, 0.05, True)
        flow[0, 0, :3] += 0.7                                   # a band that leaves the frame
        xr, mr, m_t = x[:, :, 1:], m[:, :, 1:], m[:, :, 0]
        xa, va, vm = mtb.dfpn_align_tail(dev(xr), dev(mr), dev(m_t), dev(flow))
        oxa, ova, ovm = oracle.dfpn_align_tail(xr, mr, m_t, flow)
        assert np.array_equal(host(xa), oxa) and np.array_equal(host(va), ova) and np.array_equal(host(vm), ovm)


@pytest.mark.parametrize("reduction", ["sum", "mean"])
def test_masked_l1_layouts(mtb, reduction):
    """mt_masked_l1_fwd / _bwd over the memory layouts the launcher treats differently: everything folded into one plane
    per sample (no mask / per-channel mask), frames folded only (mask shared by the channels), nothing folded (a strided
    frame view; a mask broadcast over the frames), odd sizes on the scalar path, a batch selection - against the oracle."""
    from master_thesis_b200 import ops
    r = np.random.RandomState(77)
    B, C, F, H, W = 3, 3, 4, 10, 12

    def rnd(*shape):
        return r.standard_normal(shape).astype(np.float32)

    bm = np.array([True, False, True])
    cases_ = {
        "none": (rnd(B, C, F, H, W), rnd(B, C, F, H, W), None, bm),
        "per_channel": (rnd(B, C, F, H, W), rnd(B, C, F, H, W), (r.random_sample((B, C, F, H, W)) < 0.6).astype(np.float32), None),
        "shared": (rnd(B, C, F, H, W), rnd(B, C, F, H, W), (r.random_sample((B, 1, F, H, W)) < 0.6).astype(np.float32), bm),
        "odd": (rnd(2, 3, 2, 5, 7), rnd(2, 3, 2, 5, 7), (r.random_sample((2, 1, 2, 5, 7)) < 0.5).astype(np.float32), None),
        "flow": (rnd(B, F, H, W, 2), rnd(B, F, H, W, 2), None, bm),           # (B, F, H, W, 2): C = F, F = H, P = W * 2
    }
    for key, (ya, yb, mk, sel) in cases_.items():
        a = dev(ya).requires_grad_(True)
        loss = ops.masked_l1(a, dev(yb), None if mk is None else dev(mk), None if sel is None else dev(sel),
                             reduction, 1.25)
        loss.backward()
        full = np.ones_like(ya) if mk is None else mk
        want = oracle.masked_l1(ya, yb, full, sel, reduction, 1.25)
        assert float(loss) == pytest.approx(want, rel=2e-6), key
        wg = -oracle.masked_l1_bwd(ya, yb, full, sel, reduction, 1.25)   # the oracle returns d / d y = -d / d y_hat
        assert np.abs(host(a.grad) - wg).max() <= 1e-6 * max(np.abs(wg).max(), 1e-30), key
    # strided frame view (every second frame of a longer clip): nothing can be folded
    big_a, big_b = rnd(B, C, 2 * F, H, W), rnd(B, C, 2 * F, H, W)
    mk = (r.random_sample((B, 1, F, H, W)) < 0.6).astype(np.float32)
    a = dev(big_a)[:, :, ::2]
    loss = ops.masked_l1(a, dev(big_b)[:, :, ::2], dev(mk), None, reduction, 1.0)
    want = oracle.masked_l1(big_a[:, :, ::2], big_b[:, :, ::2], mk, None, reduction, 1.0)
    assert float(loss) == pytest.approx(want, rel=2e-6)
