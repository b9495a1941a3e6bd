"""Batched clip inpainting: ops.chn_fill_lanes (composite + hole update of L target frames, one hole percentage per
lane, in place through a slot table) against ops.chn_fill at B = 1, and the batched patched CHN.inpaint_ff /
inpaint_cp against the one-frame-at-a-time loops, bit for bit."""
import contextlib
import os

import numpy as np
import pytest
import torch

import cases
from master_thesis_b200 import ops, plug, synth

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def mtb():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device")
    import master_thesis_b200 as m
    from master_thesis_b200 import _lib
    _lib.load()
    return m


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.detach().contiguous().cpu().numpy()


def _lane_inputs(seed, L, h, w):
    """nn_out, x_t (L,3,h,w), {0,1} masks m_t and v_map0 <= m_t (L,1,h,w): what the loops carry."""
    r = synth.rng(seed)
    nn_out = r.standard_normal((L, 3, h, w)).astype(np.float32)
    x_t = r.random_sample((L, 3, h, w)).astype(np.float32)
    m_t = (r.random_sample((L, 1, h, w)) < 0.3).astype(np.float32)
    v_map0 = m_t * (r.random_sample((L, 1, h, w)) < 0.5).astype(np.float32)
    return nn_out, x_t, m_t, v_map0


def _per_lane_reference(nn_out, x_t, m_t, v_map0):
    """ops.chn_fill at B = 1 on every lane's slice: [(y_comp, m_new, x_new, inp_per)]."""
    out = []
    for i in range(nn_out.shape[0]):
        mt = dev(m_t[i:i + 1])
        yc, m_new, x_new, per = ops.chn_fill(dev(nn_out[i:i + 1]), dev(x_t[i:i + 1]), 1 - mt, mt, dev(v_map0[i:i + 1]))
        out.append((host(yc)[0], host(m_new)[0], host(x_new)[0], np.float32(host(per))))
    return out


def _state(S, h, w, fill=-7.0):
    return (torch.full((S, 3, h, w), fill, device="cuda"), torch.full((S, 1, h, w), fill, device="cuda"),
            torch.full((S, 3, h, w), fill, device="cuda"), torch.full((S,), fill, device="cuda"))


# ---------------------------------------------------------------- kernel parity
@gpu
@pytest.mark.parametrize("h,w", [(16, 20), (15, 21), (48, 64)], ids=["vec4", "ragged", "wide"])
@pytest.mark.parametrize("L", [1, 3, 8])
def test_fill_lanes_equals_fill_step_per_lane(mtb, L, h, w):
    nn_out, x_t, m_t, v_map0 = _lane_inputs(100 + L + h, L, h, w)
    want = _per_lane_reference(nn_out, x_t, m_t, v_map0)
    S = L + 3
    slots = [int(s) for s in synth.rng(7 + L).permutation(S)[:L]]
    x_s, m_s, y_o, per = _state(S, h, w)
    ops.chn_fill_lanes(dev(nn_out), dev(x_t), dev(m_t), dev(v_map0), slots, x_s, m_s, y_o, per)
    got = [host(t) for t in (y_o, m_s, x_s, per)]
    for i, s in enumerate(slots):
        yc, m_new, x_new, p = want[i]
        assert np.array_equal(got[0][s], yc) and np.array_equal(got[1][s], m_new) and np.array_equal(got[2][s], x_new)
        assert got[3][s].tobytes() == p.tobytes()
    untouched = sorted(set(range(S)) - set(slots))
    for t in got:
        assert (t[untouched] == -7.0).all()


@gpu
@pytest.mark.parametrize("h,w", [(16, 20), (15, 21)], ids=["vec4", "ragged"])
def test_fill_lanes_in_place(mtb, h, w):
    """x_t / m_t as strided views of the very state slots the lanes update."""
    L = 4
    nn_out, x_t, m_t, v_map0 = _lane_inputs(31, L, h, w)
    want = _per_lane_reference(nn_out, x_t, m_t, v_map0)
    S = 2 * L
    x_s, m_s, y_o, per = _state(S, h, w)
    x_s[0::2] = dev(x_t)
    m_s[0::2] = dev(m_t)
    slots = list(range(0, S, 2))
    ops.chn_fill_lanes(dev(nn_out), x_s[0::2], m_s[0::2], dev(v_map0), slots, x_s, m_s, y_o, per)
    for i, s in enumerate(slots):
        yc, m_new, x_new, p = want[i]
        assert np.array_equal(host(y_o[s]), yc) and np.array_equal(host(m_s[s]), m_new)
        assert np.array_equal(host(x_s[s]), x_new) and host(per)[s].tobytes() == p.tobytes()
    assert (host(x_s[1::2]) == -7.0).all() and (host(m_s[1::2]) == -7.0).all()


@gpu
@pytest.mark.parametrize("h,w", [(16, 20), (15, 21)], ids=["vec4", "ragged"])
def test_fill_lanes_finalize(mtb, h, w):
    """inpaint_cp's `if float(per) < e or force: m = 0, y = y_comp` per lane, with e just above, at and just below
    one lane's percentage."""
    L = 5
    nn_out, x_t, m_t, v_map0 = _lane_inputs(47, L, h, w)
    want = _per_lane_reference(nn_out, x_t, m_t, v_map0)
    pers = [float(p) for *_, p in want]
    assert len(set(pers)) > 1
    k = int(np.argsort(pers)[L // 2])
    slots = [4, 0, 3, 1, 2]
    for e, force in ((np.nextafter(pers[k], np.inf), False), (pers[k], False), (np.nextafter(pers[k], -np.inf), False),
                     (-1.0, True), (101.0, False)):
        x_s, m_s, y_o, per = _state(L, h, w)
        ops.chn_fill_lanes(dev(nn_out), dev(x_t), dev(m_t), dev(v_map0), slots, x_s, m_s, y_o, per, (float(e), force))
        n_final = 0
        for i, s in enumerate(slots):
            yc, m_new, x_new, p = want[i]
            fin = float(p) < float(e) or force
            n_final += fin
            assert np.array_equal(host(y_o[s]), yc) and host(per)[s].tobytes() == p.tobytes()
            assert np.array_equal(host(m_s[s]), np.zeros_like(m_new) if fin else m_new)
            assert np.array_equal(host(x_s[s]), yc if fin else x_new)
        assert 0 < n_final or e < min(pers)


@gpu
def test_fill_lanes_workspace_serves_any_lane_count(mtb):
    """One zeroed workspace shared by calls of different lane counts, in the order a pass of inpaint_cp with a large
    batch meets them (a full chunk, a short remainder, a full chunk again): every call's percentages must be
    complete, whatever the previous call left in the workspace."""
    h, w = 5, 7                                             # one chunk per lane: a single CTA folds each lane
    key = ("lanes", torch.cuda.current_device(), torch.cuda.current_stream().cuda_stream)
    saved = ops._workspaces.pop(key, None)
    try:
        for i, L in enumerate((70, 5, 5, 70, 3, 130, 70)):
            nn_out, x_t, m_t, v_map0 = _lane_inputs(500 + i, L, h, w)
            x_s, m_s, y_o, per = _state(L, h, w)
            ops.chn_fill_lanes(dev(nn_out), dev(x_t), dev(m_t), dev(v_map0), list(range(L)), x_s, m_s, y_o, per)
            m_new = m_t - v_map0
            want = np.array([np.float32(m_new[k].sum()) * np.float32(100.0) / np.float32(h * w) for k in range(L)],
                            np.float32)
            assert host(per).tobytes() == want.tobytes(), "call %d (L = %d)" % (i, L)
    finally:
        ops._workspaces.pop(key, None)
        if saved is not None:
            ops._workspaces[key] = saved


@gpu
def test_fill_lanes_no_out_of_bounds_writes(mtb):
    """Every output of chn_fill_lanes and its workspace sit inside sentinel-filled buffers; ragged planes, the
    scalar and vector paths, finalisation on the device."""
    G = 256
    made = []

    def guarded(shape, sentinel=-12345.0, dtype=torch.float32):
        n = int(np.prod(shape))
        buf = torch.full((n + 2 * G,), sentinel, dtype=dtype, device="cuda")
        made.append((buf, n, sentinel))
        return buf[G:G + n].view(shape)

    Lmax = 9
    key = ("lanes", torch.cuda.current_device(), torch.cuda.current_stream().cuda_stream)
    saved = ops._workspaces.pop(key, None)
    nbytes = int(mtb._lib.load().mt_chn_fill_lanes_workspace_bytes(Lmax))
    ws = guarded((nbytes,), 0xA5, torch.uint8)
    ws.zero_()
    ops._workspaces[key] = ws
    try:
        for L, h, w, fin in ((1, 7, 9, None), (3, 15, 21, (2.0, False)), (Lmax, 17, 36, (50.0, False)),
                             (4, 16, 20, (0.0, True))):
            nn_out, x_t, m_t, v_map0 = _lane_inputs(L * 13 + w, L, h, w)
            S = L + 2
            x_s, m_s, y_o = guarded((S, 3, h, w)), guarded((S, 1, h, w)), guarded((S, 3, h, w))
            per = guarded((S,))
            ops.chn_fill_lanes(dev(nn_out), dev(x_t), dev(m_t), dev(v_map0), list(range(S - 1, S - 1 - L, -1)),
                               x_s, m_s, y_o, per, fin)
        torch.cuda.synchronize()
    finally:
        ops._workspaces.pop(key, None)
        if saved is not None:
            ops._workspaces[key] = saved
    for buf, n, sentinel in made:
        assert bool((buf[:G] == sentinel).all()) and bool((buf[G + n:] == sentinel).all()), "guard band (n=%d)" % n


# ---------------------------------------------------------------- loops
def _pick_rows(presets, key):
    """The preset of each batch row, chosen by that row's content alone (the per-row form of
    test_gpu_parity._inpaint_harness(by_content=True)): at B = 1 it is exactly what the sequential loop sees."""
    return dev(np.concatenate([presets[int(float(key[b].double().abs().sum()) * 1000.0) % len(presets)]
                               for b in range(key.shape[0])], 0))


def _harness(aligner, flows, thetas, nn_outs, batch_frames=None):
    """Stand-ins for the CHN module and its patched aligner (DFPN dense flow at frame size, DFPN flow at 256 x 256
    resized in the warp, CPN theta); every CNN call is logged as (rows, per-row content keys)."""
    log = []

    class _DFPNLike(object):
        align = plug.dfpn_align

        def __call__(self, x_target, m_target, x_refs, m_refs):
            return None, None, None, _pick_rows(flows, m_target + x_refs[:, :1, 0])

    class _DFPNLowres(_DFPNLike):
        def _mt_b200_flow_256(self, x_target, m_target, x_refs, m_refs):
            return _pick_rows(flows, m_target + x_refs[:, :1, 0])

    class _CPNLike(object):
        align = plug.cpn_align

        def A_Encoder(self, x, m):
            return torch.cat([x, m], 1)

        def A_Regressor(self, target_feats, ref_feats):
            return _pick_rows(thetas, target_feats[:, 3:] + ref_feats[:, :1])

    class _CHNLike(object):
        forward = plug.chn_forward
        inpaint_ff = plug.chn_inpaint_ff
        inpaint_cp = plug.chn_inpaint_cp
        get_indexes_ff = staticmethod(cases.get_indexes_ff)

        def __init__(self):
            self.model_aligner = {"dense": _DFPNLike, "lowres": _DFPNLowres, "cpn": _CPNLike}[aligner]()
            if batch_frames is not None:
                self.mt_b200_batch_frames = batch_frames

        def nn(self, inp):
            log.append(int(inp.shape[0]))
            return _pick_rows(nn_outs, inp[:, 6:])

        def __call__(self, *a):
            return self.forward(*a)

    return _CHNLike(), log


def _clip(seed, n, h, w, no_hole=()):
    x, m, _ = synth.frames(seed, 1, n, h, w)
    x, m = x[0].copy(), m[0].copy()
    for t in no_hole:
        m[:, t] = 0.0
    x = x * (1 - m)
    k = 11
    flows = [synth.dense_flow(seed + 10 + i, 1, 1, h, w, 0.05, True) for i in range(k)]
    flows256 = [synth.dense_flow(seed + 30 + i, 1, 1, 256, 256, 0.05, True) for i in range(k)]
    thetas = [synth.thetas(seed + 50 + i, 1, 0.1) for i in range(k)]
    nn_outs = [synth.nn_output(seed + 70 + i, 1, h, w) for i in range(k)]
    return x, m, flows, flows256, thetas, nn_outs


FF_CLIPS = {
    "ff_n4": dict(cases.INPAINT_CASES["ff_n4"]),
    "ff_n6_long": dict(cases.INPAINT_CASES["ff_n6_long"]),
    "ff_n12": dict(seed=96, n=12, h=18, w=26, e=0.05),
    "ff_n5_256": dict(seed=97, n=5, h=256, w=256, e=0.2),
}


def _run(algo, aligner, clip, batch_frames, **kw):
    x, m, flows, flows256, thetas, nn_outs = clip
    chn, log = _harness(aligner, flows256 if aligner == "lowres" else flows, thetas, nn_outs, batch_frames)
    fn = chn.inpaint_ff if algo == "ff" else chn.inpaint_cp
    y = fn(dev(x), dev(m), **kw)
    return host(y), log


@gpu
@pytest.mark.parametrize("aligner", ["dense", "lowres", "cpn"])
@pytest.mark.parametrize("lanes", [2, 3, "n"])
@pytest.mark.parametrize("name", sorted(FF_CLIPS))
def test_inpaint_ff_batched_equals_sequential(mtb, name, lanes, aligner):
    spec = FF_CLIPS[name]
    if aligner == "lowres" and spec["h"] == 256:
        pytest.skip("256 x 256 frames take the DFPN's own flow")
    n = spec["n"]
    L = n if lanes == "n" else lanes
    clip = _clip(spec["seed"], n, spec["h"], spec["w"])
    kw = dict(s=1, D=20, e=spec.get("e", 1))
    y1, log1 = _run("ff", aligner, clip, None, **kw)
    yL, logL = _run("ff", aligner, clip, L, **kw)
    assert np.array_equal(yL, y1)
    assert set(log1) == {1} and sum(logL) == len(log1)     # CNN rows == sequential fill steps
    assert max(logL) == min(L, n) and len(logL) < len(log1)
    if "long" in name or name == "ff_n12":
        assert len(log1) > n                                 # targets really iterate (lane refill for L < n)


@gpu
@pytest.mark.parametrize("aligner", ["dense", "cpn"])
@pytest.mark.parametrize("lanes", [2, "n"])
@pytest.mark.parametrize("N", [3, 5])
@pytest.mark.parametrize("s", [1, 2, 3])
def test_inpaint_cp_batched_equals_sequential(mtb, s, N, lanes, aligner, monkeypatch):
    """e is placed between the hole percentages of two first steps of pass 0 (which no choice of e changes: every
    target starts from the clip), so in the unforced first pass some lanes finalise on `per < e` on the device and
    others carry their hole on; the fill launches are watched to show that both happen."""
    n, h, w = 11, 16, 20
    clip = _clip(98 + s, n, h, w, no_hole=(2, 7))
    L = n if lanes == "n" else lanes
    steps = []                                      # (slot, inp_per, forced) of every lane of every unforced launch
    fill_lanes = ops.chn_fill_lanes

    def watched(nn_out, x_t, m_t, v_map0, slots, x_state, m_state, y_out, per_out, finalize=None):
        fill_lanes(nn_out, x_t, m_t, v_map0, slots, x_state, m_state, y_out, per_out, finalize)
        if finalize is not None and not finalize[1]:
            steps.extend((sl, p, finalize[0]) for sl, p in zip(slots, per_out[slots].tolist()))
    monkeypatch.setattr(ops, "chn_fill_lanes", watched)

    _run("cp", aligner, clip, L, N=N, s=s, e=-1.0)  # probe: nothing finalises before the forced passes
    first, seen = [], set()
    for sl, p, _ in steps:
        if sl not in seen:
            seen.add(sl)
            first.append(p)
    levels = sorted(set(first))
    assert len(levels) >= 2, first
    k = len(levels) // 2
    e = (levels[k - 1] + levels[k]) / 2.0           # some first steps fall below e, others do not
    del steps[:]
    y1, log1 = _run("cp", aligner, clip, None, N=N, s=s, e=e)
    yL, logL = _run("cp", aligner, clip, L, N=N, s=s, e=e)
    assert np.array_equal(yL, y1)
    assert set(log1) == {1} and sum(logL) == len(log1) and max(logL) <= L
    assert len(logL) < len(log1)
    assert any(p < e for _, p, _ in steps) and any(not p < e for _, p, _ in steps)   # early finalisation exercised


@gpu
@pytest.mark.parametrize("algo", ["ff", "cp"])
def test_default_keeps_the_sequential_call_sequence(mtb, algo, monkeypatch):
    """Knob absent, 1 on the module, or 1 in the environment: one row per CNN call, the same calls in the same
    order (the content keys of every call are logged, not just the counts)."""
    spec = FF_CLIPS["ff_n6_long"]
    clip = _clip(spec["seed"], spec["n"], spec["h"], spec["w"])
    kw = dict(s=1, D=20, e=spec["e"]) if algo == "ff" else dict(N=3, s=1, e=0.5)
    keys = []

    def run(batch_frames):
        x, m, flows, _, thetas, nn_outs = clip
        chn, log = _harness("dense", flows, thetas, nn_outs, batch_frames)
        seen = []
        nn = chn.nn
        chn.nn = lambda inp: (seen.append(host(inp).tobytes()), nn(inp))[1]
        y = (chn.inpaint_ff if algo == "ff" else chn.inpaint_cp)(dev(x), dev(m), **kw)
        keys.append(seen)
        return host(y), log

    monkeypatch.delenv("MT_INPAINT_BATCH_FRAMES", raising=False)
    y0, log0 = run(None)
    y1, log1 = run(1)
    monkeypatch.setenv("MT_INPAINT_BATCH_FRAMES", "1")
    y2, log2 = run(None)
    assert set(log0) == {1} and log0 == log1 == log2
    assert keys[0] == keys[1] == keys[2]
    assert np.array_equal(y0, y1) and np.array_equal(y0, y2)
    monkeypatch.setenv("MT_INPAINT_BATCH_FRAMES", "4")
    y4, log4 = run(None)
    assert np.array_equal(y4, y0) and max(log4) > 1


# ---------------------------------------------------------------- CPU
def test_fill_lanes_rejects_bad_slots_before_any_launch(monkeypatch):
    from master_thesis_b200 import _lib

    def no_launch(*a, **k):
        raise AssertionError("launched")
    monkeypatch.setattr(_lib, "call", no_launch)
    L, S, h, w = 3, 5, 4, 4
    lanes3, lanes1 = torch.zeros(L, 3, h, w), torch.zeros(L, 1, h, w)
    state = (torch.zeros(S, 3, h, w), torch.zeros(S, 1, h, w), torch.zeros(S, 3, h, w), torch.zeros(S))
    for slots, msg in (([0, 1, 1], "duplicate"), ([0, 1, 5], "out of range"), ([-1, 0, 1], "out of range"),
                       ([0, 1], "2 slots for 3 lanes")):
        with pytest.raises(ValueError, match=msg):
            ops.chn_fill_lanes(lanes3, lanes3, lanes1, lanes1, slots, *state)
    with pytest.raises(RuntimeError, match="CUDA tensors required"):       # good slots: then the device check
        ops.chn_fill_lanes(lanes3, lanes3, lanes1, lanes1, [4, 0, 2], *state)


def test_batch_frames_knob(monkeypatch):
    class _M(object):
        pass
    monkeypatch.delenv("MT_INPAINT_BATCH_FRAMES", raising=False)
    assert plug._batch_frames(_M()) == 1
    monkeypatch.setenv("MT_INPAINT_BATCH_FRAMES", "6")
    assert plug._batch_frames(_M()) == 6
    mod = _M()
    mod.mt_b200_batch_frames = 3
    assert plug._batch_frames(mod) == 3
    mod.mt_b200_batch_frames = 0
    assert plug._batch_frames(mod) == 1


def test_batched_path_applies_only_with_a_patched_aligner(monkeypatch):
    monkeypatch.delenv("MT_INPAINT_BATCH_FRAMES", raising=False)

    def chn(align, batch_frames):
        aligner = type("A", (), {"align": align})()
        m = type("C", (), {})()
        m.model_aligner = aligner
        if batch_frames is not None:
            m.mt_b200_batch_frames = batch_frames
        return m
    assert plug._lanes_grid(chn(plug.dfpn_align, None), 8) is None            # default: the sequential loops
    assert plug._lanes_grid(chn(plug.dfpn_align, 1), 8) is None
    assert plug._lanes_grid(chn(plug.dfpn_align, 4), 8) is plug._dfpn_grid
    assert plug._lanes_grid(chn(plug.cpn_align, 4), 8) is plug._cpn_grid
    assert plug._lanes_grid(chn(plug.dfpn_align, 4), 1) is None               # n < 2
    assert plug._lanes_grid(chn(lambda *a: None, 4), 8) is None               # a foreign aligner


def test_patch_rebinds_the_same_plug_points():
    import types
    mt = types.SimpleNamespace()
    for mod, cls, attr, _, static in plug._PATCHES:
        m = getattr(mt, mod, None) or types.SimpleNamespace()
        setattr(mt, mod, m)
        k = getattr(m, cls, None) or type(cls, (), {})
        setattr(m, cls, k)
        setattr(k, attr, staticmethod(lambda *a: "orig") if static else (lambda *a: "orig"))
    names = plug.patch(mt)
    try:
        assert len(names) == len(set(names)) == 18
        assert mt.model_chn.CHN.inpaint_ff is plug.chn_inpaint_ff
        assert mt.model_chn.CHN.inpaint_ip is plug.chn_inpaint_ip
        assert mt.model_chn.CHN.inpaint_cp is plug.chn_inpaint_cp
        assert not hasattr(mt.model_chn.CHN, "mt_b200_batch_frames")       # opt-in: patch() sets no knob
    finally:
        plug.unpatch(mt)
    assert mt.model_chn.CHN.inpaint_cp(None) == "orig"
