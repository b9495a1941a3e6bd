"""CPU-side tests: the C-ABI library builds, loads and exports every declared
symbol; the host mirrors fail loudly without a GPU; patch() rebinds the
reference plug points; the rank partitioning is exact (gloo, world_size 2)."""
import ctypes
import os
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

import cases
import oracle
from master_thesis_b200 import _lib, build, ops, plug, shard

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    build.build_library()
    return _lib.load()


def test_library_exports_every_declared_symbol(lib):
    protos = _lib.parse_header()
    assert len(protos) >= 24
    out = subprocess.check_output(["nm", "-D", "--defined-only", _lib.LIB_PATH], text=True)
    exported = {ln.split()[-1] for ln in out.splitlines() if " T " in ln}
    assert set(protos) <= exported
    assert exported == set(protos), "exported but undeclared: %s" % (exported - set(protos))
    assert lib.mt_version() >= 100
    assert lib.mt_workspace_bytes() > 0
    assert lib.mt_cm_workspace_bytes(8, 128, 5, 64, 64) > 0


def test_library_is_sm100a_only():
    out = subprocess.check_output(["cuobjdump", "--list-elf", _lib.LIB_PATH], text=True)
    archs = {ln.split(".")[-2] for ln in out.splitlines() if ".cubin" in ln}
    assert archs == {"sm_100a"}, archs


def test_bad_arguments_return_error_codes(lib):
    assert lib.mt_mask_out(None, 10, None, None) == -1
    assert "mt_mask_out" in _lib.last_error()
    assert lib.mt_cm_match_fwd(None, None, None, None, None, None, 1, 1, 2, 4, 4, 16, 16, None) == -1
    with pytest.raises(RuntimeError):
        _lib.call("mt_corr4d_fwd", None, None, None, None, None, None, 0, 1, 1, 1, 16, None)


def test_missing_library_fails_loudly(monkeypatch):
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libmt_b200.so")
    with pytest.raises(RuntimeError, match="no CPU"):
        _lib.load()


def test_ops_reject_cpu_tensors():
    x = torch.zeros(1, 3, 1, 4, 4)
    with pytest.raises(RuntimeError, match="CUDA tensors required"):
        ops.warp_fwd(x, x[:, :1], torch.zeros(1, 1, 4, 4, 2))
    with pytest.raises(RuntimeError, match="CUDA tensors required"):
        plug.LossesUtils.masked_l1(x, x, x)
    with pytest.raises(RuntimeError, match="CUDA tensors required"):
        plug.CM_Module()(torch.zeros(1, 4, 3, 4, 4), torch.zeros(1, 1, 16, 16), torch.zeros(1, 1, 2, 16, 16))


def test_product_never_imports_oracle():
    for root, _, files in os.walk(os.path.join(ROOT, "master_thesis_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(root, f)).read()
                assert "import oracle" not in text and "from oracle" not in text, f
                assert "mt_oracle" not in text and "libmt_oracle" not in text, f


def _mock_reference():
    mt = types.SimpleNamespace()
    for mod, cls, attr, _, static in plug._PATCHES:
        m = getattr(mt, mod, None) or types.SimpleNamespace()
        setattr(mt, mod, m)
        k = getattr(m, cls, None) or type(cls, (), {})
        setattr(m, cls, k)
        fn = (lambda *a, **kw: "orig")
        setattr(k, attr, staticmethod(fn) if static else fn)
    mt.FlowsUtils = mt.utils.FlowsUtils      # the package re-exports utils' classes at its top level
    return mt


def test_patch_rebinds_and_unpatch_restores():
    mt = _mock_reference()
    names = plug.patch(mt)
    assert "model_cpn.CPN.align" in names and "utils.FlowsUtils.align_set" in names
    assert mt.model_cpn.CPN.align is plug.cpn_align
    assert mt.model_dfpn.DFPN.align is plug.dfpn_align
    assert mt.utils.FlowsUtils.align_set is plug.FlowsUtils.align_set
    assert mt.FlowsUtils.align_set is plug.FlowsUtils.align_set      # the package-level alias too
    assert mt.model_chn.CHN.forward is plug.chn_forward
    plug.patch(mt)          # idempotent
    plug.unpatch(mt)
    assert mt.utils.FlowsUtils.align_set() == "orig"
    assert mt.FlowsUtils.align_set() == "orig"
    assert mt.model_cpn.CPN.align(None) == "orig"


def test_block_ranges_partition_exactly():
    for n in (0, 1, 7, 32, 33, 256):
        for world in (1, 2, 3, 4, 8):
            got = []
            for r in range(world):
                lo, hi = shard.block_range(n, r, world)
                got += list(range(lo, hi))
                assert hi - lo in (n // world, n // world + 1)
            assert got == list(range(n))
    assert shard.frame_shard(2, 3, 1, 2) == [(1, 0), (1, 1), (1, 2)]
    assert shard.frame_shard_groups(2, 3, 0, 4) == {0: (0, 2)}
    with pytest.raises(ValueError):
        shard.block_range(4, 2, 2)


_WORKER = r"""
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, 'tests', 'golden'))
import cases, oracle
from master_thesis_b200 import shard
dist.init_process_group('gloo', init_method='tcp://127.0.0.1:{port}', rank=int(sys.argv[1]), world_size=2)
rank, world = dist.get_rank(), dist.get_world_size()
x, m, m_t, flow = cases.warp_inputs(cases.WARP_CASES['smooth_f4'])
b, c, f, h, w = x.shape
full = oracle.dfpn_align_tail(x, m, m_t, flow)
# each rank computes only its (b, f) block, grouped per sample as the GPU path launches it
mine = np.zeros((b * f, c + 2, h, w), np.float32)
for bi, (f0, f1) in shard.frame_shard_groups(b, f, rank, world).items():
    xa, va, vm = oracle.dfpn_align_tail(x[bi:bi+1, :, f0:f1], m[bi:bi+1, :, f0:f1], m_t[bi:bi+1], flow[bi:bi+1, f0:f1])
    for k, fi in enumerate(range(f0, f1)):
        mine[bi * f + fi, :c] = xa[0, :, k]; mine[bi * f + fi, c] = va[0, 0, k]; mine[bi * f + fi, c + 1] = vm[0, 0, k]
t = torch.from_numpy(mine)
dist.all_reduce(t)          # test-only gather (blocks are disjoint); the data path has no collective
got = t.numpy()
ref = np.concatenate([full[0].transpose(0, 2, 1, 3, 4).reshape(b * f, c, h, w), full[1].reshape(b * f, 1, h, w), full[2].reshape(b * f, 1, h, w)], 1)
assert np.array_equal(got, ref), 'sharded result differs'
# CM shards by sample only
cf, vt, va = cases.cm_inputs(cases.CM_CASES['edge'])
lo, hi = shard.batch_shard(cf.shape[0], rank, world)
part = np.zeros((cf.shape[0],) + oracle.cm_module(cf[:1], vt[:1], va[:1])[0].shape[1:], np.float32)
if hi > lo:
    part[lo:hi] = oracle.cm_module(cf[lo:hi], vt[lo:hi], va[lo:hi])[0]
t = torch.from_numpy(part); dist.all_reduce(t)
assert np.array_equal(t.numpy(), oracle.cm_module(cf, vt, va)[0])
dist.destroy_process_group()
print('rank', rank, 'ok')
"""


def test_two_rank_sharding_gloo(tmp_path):
    """world_size 2 on CPU (gloo): per-rank (b, f) blocks reproduce the unsharded result."""
    oracle.build()
    port = 29500 + (os.getpid() % 2000)
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT, port=port))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
        assert "ok" in o


def test_recorded_plan_owns_its_buffers():
    """Buffers allocated by the operators while recording must stay alive with the Plan:
    torch.cuda.graph() empties the allocator cache, which unmapped freed temporaries that a
    plan still wrote to (an illegal address in bench.py's cfg5)."""
    import weakref
    t = torch.zeros(4)
    assert _lib.keep(t) is t                      # no-op outside a recording
    with _lib.record() as plan:
        a = ops._empty(8)
        b = ops._contig(torch.zeros(4, 4).t())    # non-contiguous: a copy is made and kept
        c = ops._contig(torch.zeros(4))           # already contiguous: kept as it is (a replay reads its pointer)
    refs = [weakref.ref(a), weakref.ref(b), weakref.ref(c)]
    assert len(plan.keep) == 3 and plan.keep[0] is a and plan.keep[1] is b and plan.keep[2] is c
    del a, b, c
    assert all(r() is not None for r in refs)     # the plan keeps them alive
    del plan
    assert all(r() is None for r in refs)


def test_masked_l1_layout_of_broadcast_masks():
    """ADVICE r1: the (B, C, F, P) decomposition never expands a mask into the 'sum' denominator: broadcast axes
    become stride 0 and `repeat` counts how often every element of the mask as given is visited."""
    y4 = torch.zeros(3, 4, 6, 8)
    (a, b_, m), B, C, F, P, mask_c, repeat = ops._l1_layout(y4, y4, torch.zeros(3, 1, 6, 8))
    assert (B, C, F, P, mask_c, repeat) == (3, 4, 1, 48, 1, 1) and m[1:] == (48, 0, 0) and a[1:] == (192, 48, 0)
    y5 = torch.zeros(3, 4, 5, 6, 8)
    (_, _, m), B, C, F, P, mask_c, repeat = ops._l1_layout(y5, y5, torch.zeros(3, 1, 1, 6, 8))
    assert (B, C, F, P, mask_c, repeat) == (3, 4, 5, 48, 1, 5) and m[1:] == (48, 0, 0)
    (_, _, m), *_, mask_c, repeat = ops._l1_layout(y5, y5, torch.zeros(1, 4, 5, 6, 8))
    assert (mask_c, repeat) == (4, 3) and m[1:] == (0, 240, 48)
    (_, _, m), *_, mask_c, repeat = ops._l1_layout(y5, y5, torch.zeros(3, 1, 5, 1, 1))
    assert (mask_c, repeat) == (1, 48) and m[0].shape == (3, 1, 5, 6, 8) and m[1:] == (240, 0, 48)
    (_, _, m), *_, mask_c, repeat = ops._l1_layout(y5, y5, torch.zeros(3, 4, 5, 6, 8))
    assert (mask_c, repeat) == (4, 1)
    # the flows of DFPN.compute_loss: (B, F, h, w, 2) against a mask of ones of the same shape
    fl = torch.zeros(2, 4, 16, 16, 2)
    (a, _, m), B, C, F, P, mask_c, repeat = ops._l1_layout(fl, fl, torch.ones_like(fl))
    assert (B, C, F, P, mask_c, repeat) == (2, 4, 16, 32, 4, 1)
    with pytest.raises(RuntimeError, match="broadcast"):
        ops._l1_layout(y5, y5, torch.zeros(3, 2, 5, 6, 8))
    # mask=None stands for torch.ones_like(y_hat): no tensor at all, the kernels take mask = NULL as all ones
    (_, _, m), B, C, F, P, mask_c, repeat = ops._l1_layout(y5, y5, None)
    assert (mask_c, repeat) == (4, 1) and m == (None, 0, 0, 0)


def test_deferred_align_is_transparent():
    """An xs_aligned handle of the patched DFPN._train_val_wrapper behaves like the aligned tensor for anyone
    who touches it (here: materialisation is stubbed, no GPU involved)."""
    d = plug.DeferredAlign("x", "v", "flow")
    d._done = (torch.arange(6.0).reshape(2, 3), None)
    assert d.size() == (2, 3) and float(torch.sum(d)) == 15.0 and float(d.double().sum()) == 15.0
    assert torch.equal(torch.cat([d, d]), torch.cat([d._done[0], d._done[0]]))
