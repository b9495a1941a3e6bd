"""Batched clip inpainting on 480 x 854 clips: the patched CHN.inpaint_ff / inpaint_cp one target frame at a time
against L target frames per fill step (plug._batch_frames), and the fill kernel alone.

Loop level: clips of 8 and 32 frames, CNN stand-ins at zero cost as in bench.py's Cfg4.loop_stats (the DFPN stand-in
hands out a 256 x 256 flow per row, the RRDBNet a preset output per row).  Every number is wall clock around work that
ends in a device synchronise, after a warm-up pass; host reads and CNN calls are counted in a separate pass.
Kernel level: CUDA events around graph replays of one mt_chn_fill_lanes launch at L = 8 against 8 launches of
mt_chn_fill_step at B = 1 on the same data, with the algorithmic bytes (64 B per pixel and lane, as Cfg4.calls
counts them) as a share of the copy bandwidth measured in the same run.  The effect with the real RRDBNet / DFPN is
not measured here.

    python tools/gpu/time_inpaint_batched.py [out.json]
"""
import contextlib
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from master_thesis_b200 import _lib, ops, plug, synth    # noqa: E402

H, W = 480, 854
REPS = 3


def power_limit():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                                        str(torch.cuda.current_device())], text=True, timeout=30).strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def copy_bandwidth():
    """Device-to-device copy of 2 GiB: read + write bytes over time, the best of 10 (GB/s)."""
    a = torch.empty(2 ** 29, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    a.fill_(1.0)
    best = 0.0
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        torch.cuda.synchronize()
        best = max(best, 2 * a.numel() * 4 / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    del a, b
    return best


@contextlib.contextmanager
def count_host_reads(counter):
    """Counts the device->host reads the loops make (float(), bool(), .item(), .tolist() of CUDA tensors)."""
    names = ("__float__", "__bool__", "item", "tolist")
    saved = {n: getattr(torch.Tensor, n) for n in names}

    def wrap(fn):
        def f(self, *a, **k):
            if self.is_cuda:
                counter[0] += 1
            return fn(self, *a, **k)
        return f
    for n in names:
        setattr(torch.Tensor, n, wrap(saved[n]))
    try:
        yield
    finally:
        for n in names:
            setattr(torch.Tensor, n, saved[n])


def stand_ins(flow, nn_o):
    calls = []

    class _DFPN(object):
        align = plug.dfpn_align

        def __call__(self, x_target, *a):
            return None, None, None, flow[:x_target.shape[0]]

    class _CHN(object):
        forward = plug.chn_forward
        inpaint_ff = plug.chn_inpaint_ff
        inpaint_cp = plug.chn_inpaint_cp

        def __init__(self):
            self.model_aligner = _DFPN()

        @staticmethod
        def get_indexes_ff(t, n_frames, s=1, D=20):
            return sorted((i for i in range(n_frames) if i != t), key=lambda i: abs(i - t))[:D]

        def nn(self, inp):
            calls.append(inp.shape[0])
            return nn_o[:inp.shape[0]]

        def __call__(self, *a):
            return self.forward(*a)

    return _CHN, calls


def loop_rows(n, lmax):
    x, m, _ = synth.frames(77, 1, n, H, W)
    x, m = torch.from_numpy(x[0]).cuda(), torch.from_numpy(m[0]).cuda()
    flow = torch.from_numpy(synth.dense_flow(78, 1, 1, 256, 256, 0.03, True)).cuda().expand(lmax, -1, -1, -1, -1)
    nn_o = torch.from_numpy(synth.nn_output(79, 1, H, W)).cuda().expand(lmax, -1, -1, -1)
    flow, nn_o = flow.contiguous(), nn_o.contiguous()
    cls, calls = stand_ins(flow, nn_o)
    runs = [("ff", "sequential, sync_every 1", dict(mt_b200_sync_every=1)),
            ("ff", "sequential, sync_every 8", dict(mt_b200_sync_every=8))]
    runs += [("ff", "batched, L = %d" % L, dict(mt_b200_batch_frames=L)) for L in (4, 8, 32)]
    runs += [("cp", "sequential", {})]
    runs += [("cp", "batched, L = %d" % L, dict(mt_b200_batch_frames=L)) for L in (4, 8, 32)]
    rows, ref = [], {}
    for algo, label, knobs in runs:
        chn = cls()
        for k, v in knobs.items():
            setattr(chn, k, v)

        def run():
            if algo == "ff":
                return chn.inpaint_ff(x, m, s=1, D=20, e=1)
            return chn.inpaint_cp(x.clone(), m.clone(), N=20, s=1, e=1)
        y = run()                                   # warm-up
        torch.cuda.synchronize()
        reads = [0]
        del calls[:]
        with count_host_reads(reads):
            run()
        torch.cuda.synchronize()
        n_calls, n_rows = len(calls), sum(calls)
        t0 = time.perf_counter()
        for _ in range(REPS):
            run()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / REPS
        same = bool(torch.equal(y, ref[algo])) if algo in ref else True
        ref.setdefault(algo, y)
        rows.append(dict(frames=n, algo=algo, run=label, target_frames_per_sec=round(n / dt, 1),
                         ms_per_clip=round(dt * 1e3, 2), fill_steps_per_target=round(n_rows / n, 3),
                         host_reads_per_target=round(reads[0] / n, 3), cnn_calls_per_clip=n_calls,
                         equal_to_sequential=same))
        print(json.dumps(rows[-1]), flush=True)
    return rows


def kernel_rows(bw, L=8):
    """Graph replays of one mt_chn_fill_lanes launch (L lanes) against L mt_chn_fill_step launches at B = 1."""
    P = H * W
    sets = []
    for i in range(2):          # two sets (2 x 8 lanes x 64 B x 410 k px = 420 MB) rotate: no L2 reuse between passes
        nn_out = torch.randn(L, 3, H, W, device="cuda")
        x_t = torch.rand(L, 3, H, W, device="cuda")
        m_t = (torch.rand(L, 1, H, W, device="cuda") < 0.1).float()
        v_map0 = m_t * (torch.rand(L, 1, H, W, device="cuda") < 0.5).float()
        sets.append((nn_out, x_t, m_t, v_map0, 1 - m_t))     # v_t of the B = 1 step, made outside the timing
    s = torch.cuda.Stream()
    x_s = torch.empty(L, 3, H, W, device="cuda")
    m_s = torch.empty(L, 1, H, W, device="cuda")
    y_o = torch.empty(L, 3, H, W, device="cuda")
    per = torch.empty(L, device="cuda")
    slots = torch.arange(L, dtype=torch.int32, device="cuda")
    with torch.cuda.stream(s):
        ws_l = ops.zeroed_scratch(x_s, "lanes", int(_lib.load().mt_chn_fill_lanes_workspace_bytes(L)))
        ws_1 = ops.reduce_workspace(x_s)
    torch.cuda.synchronize()

    def lanes(d):
        nn_out, x_t, m_t, v_map0, _ = d
        _lib.call("mt_chn_fill_lanes", ops._ptr(nn_out), ops._ptr(x_t), 3 * P, P, ops._ptr(m_t), P, ops._ptr(v_map0),
                  P, ops._ptr(slots), ops._ptr(y_o), 3 * P, P, ops._ptr(m_s), P, ops._ptr(x_s), 3 * P, P,
                  ops._ptr(per), ops._ptr(ws_l), L, P, 0, 1.0, 0, ops._stream(nn_out))

    def steps(d):
        nn_out, x_t, m_t, v_map0, v_t = d
        for i in range(L):
            _lib.call("mt_chn_fill_step", ops._ptr(nn_out[i]), ops._ptr(x_t[i]), 3 * P, P, ops._ptr(v_t[i]), P,
                      ops._ptr(m_t[i]), P, ops._ptr(v_map0[i]), P, ops._ptr(y_o[i]), ops._ptr(m_s[i]),
                      ops._ptr(x_s[i]), ops._ptr(per[i:]), ops._ptr(ws_1), 1, P, ops._stream(nn_out))

    graphs = {}
    for name, fn in (("lanes", lanes), ("steps", steps)):
        for i, d in enumerate(sets):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.stream(s):
                fn(d)                               # warm-up outside the capture
            torch.cuda.synchronize()
            with torch.cuda.graph(g, stream=s):
                fn(d)
            graphs[(name, i)] = g
    torch.cuda.synchronize()
    reps, out = 200, {}
    for name in ("lanes", "steps"):
        for i in range(4):
            graphs[(name, i % 2)].replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(reps):
            graphs[(name, i % 2)].replay()
        e1.record()
        torch.cuda.synchronize()
        out[name] = e0.elapsed_time(e1) * 1e3 / reps
    nbytes = 64 * P * L
    rows = []
    for name, label in (("lanes", "mt_chn_fill_lanes, L = %d, one launch" % L),
                        ("steps", "%d x mt_chn_fill_step, B = 1" % L)):
        us = out[name]
        rows.append(dict(call=label, us=round(us, 1), bytes=nbytes, GBps=round(nbytes / (us * 1e-6) / 1e9, 1),
                         share_of_copy_bw=round(nbytes / (us * 1e-6) / 1e9 / bw, 3)))
        print(json.dumps(rows[-1]), flush=True)
    return rows


def main():
    if not torch.cuda.is_available():
        raise SystemExit("time_inpaint_batched.py measures on a CUDA device; none is visible")
    torch.manual_seed(0)
    bw = copy_bandwidth()
    with torch.no_grad():
        loops = loop_rows(8, 32) + loop_rows(32, 32)
        kern = kernel_rows(bw)
    doc = dict(device=torch.cuda.get_device_name(), power_limit=power_limit(), copy_GBps=round(bw, 1),
               frame=[H, W], loop_reps=REPS,
               loop_note="CNN stand-ins at zero cost (DFPN: one 256x256 flow per row, RRDBNet: a preset per row); "
                         "ff with s=1, D=20, e=1; cp with s=1, N=20, e=1; the effect with the real RRDBNet / DFPN "
                         "is not measured",
               loop=loops, kernel=kern)
    text = json.dumps(doc, indent=1)
    print(text)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
