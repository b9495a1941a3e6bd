"""Mixed-precision DFPN aligner: the correlation and warp kernels reading half VGG features / flows natively, against
the fp32 kernels, and against what a user would otherwise write under autocast (an eager ``.float()`` of the half
operand, then the fp32 kernel).

Arms, per workload:
  fp32       fp32 operand, the fp32 entry point
  <dt>       fp16 / bf16 operand read by the *_dt entry point
  <dt>+cast  the same half operand copied to fp32 by an eager cast, then the fp32 entry point
Workloads: corr4d_vgg (C = 512, 16 x 16, masked) at 32 and 128 frames; the low-resolution warp + CNN-input pack of the
inpainting step (256 x 256 flow, 480 x 854 frames) at B = 1 and L = 8; the dense warp at 256 x 256 with 32 and 128
frames.

Every arm is one CUDA graph of REPS passes over K input sets whose total size exceeds twice the 126 MB L2, so each
pass reads its operands from HBM.  CUDA events around graph replays; the arms alternate, ROUNDS times, and the median
per arm is reported.  The fp32 arm's operand is the half operand widened.  Outputs are compared in the same run: the
warp arms bit for bit; the half correlation against the fp32 (tf32) kernel on the widened features within 2e-3 (tf32
rounds the operands, the half kernel only the result).

    python tools/gpu/time_dfpn_amp.py [out.json]
"""
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from master_thesis_b200 import _lib, ops    # noqa: E402

L2_BYTES = 126 * 2 ** 20
REPS = 4
ROUNDS = 7
HALVES = {"fp16": torch.float16, "bf16": torch.bfloat16}
FLAGS = ops.ALIGN_CORNERS | ops.VIS_FROM_MASK


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                                       "-i", str(torch.cuda.current_device())], text=True, timeout=30).strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except (OSError, subprocess.SubprocessError, ValueError):
        return {"name": torch.cuda.get_device_name(), "power_limit": "unknown", "max_sm_clock": "unknown"}


def n_sets(bytes_per_set):
    return max(2, -(-2 * L2_BYTES // bytes_per_set) + 1)


def nbytes(*ts):
    return sum(t.numel() * t.element_size() for t in ts if t is not None)


def corr_sets(b, f, dt):
    g = torch.Generator(device="cuda").manual_seed(b * 10 + f)
    one = nbytes(torch.empty((b, 512, f + 1, 16, 16), dtype=dt)) + b * f * 65536 * 4
    sets = []
    for _ in range(n_sets(one)):
        ft = torch.randn((b, 512, 16, 16), device="cuda", generator=g).to(dt)
        fr = torch.randn((b, 512, f, 16, 16), device="cuda", generator=g).to(dt)
        mt = (torch.rand((b, 1, 64, 64), device="cuda", generator=g) < 0.3).float()
        mr = (torch.rand((b, 1, f, 64, 64), device="cuda", generator=g) < 0.3).float()
        sets.append((ft, mt, fr, mr))
    return sets


def warp_sets(b, f, h, w, gh, gw, pack, dt):
    g = torch.Generator(device="cuda").manual_seed(b * 7 + h)
    sets = []
    one = b * f * (3 + 1) * h * w * 4 + b * f * gh * gw * 2 * 4 + b * f * (9 if pack else 5) * h * w * 4
    for _ in range(n_sets(one)):
        x = torch.rand((b, 3, f, h, w), device="cuda", generator=g)
        m = (torch.rand((b, 1, f, h, w), device="cuda", generator=g) < 0.1).float()
        mt = (torch.rand((b, 1, h, w), device="cuda", generator=g) < 0.1).float()
        base = torch.stack(torch.meshgrid(torch.linspace(-1, 1, gh, device="cuda"), torch.linspace(-1, 1, gw, device="cuda"),
                                          indexing="ij")[::-1], -1)
        flow = (base + 0.03 * torch.randn((b, f, gh, gw, 2), device="cuda", generator=g)).to(dt)
        xt = torch.rand((b, 3, h, w), device="cuda", generator=g)
        sets.append((x, m, flow, mt, xt, 1 - mt))
    return sets


def corr_call(s, cast):
    ft, mt, fr, mr = s
    if cast:
        ft, fr = ft.float(), fr.float()
    return ops.corr4d_vgg(ft, mt, fr, mr)


def warp_call(pack):
    def call(s, cast):
        x, m, flow, mt, xt, vt = s
        if cast:
            flow = flow.float()
        if pack:
            return ops.warp_pack_fwd(x, m, flow, mt, xt, vt, FLAGS)[:2]
        return ops.warp_fwd(x, m, flow, mt, FLAGS)
    return call


def graph_of(fn, sets, cast):
    outs = []
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for st in sets:           # warm-up: module load, tensor maps, allocator
            fn(st, cast)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(REPS):
            outs = [fn(st, cast) for st in sets]
    return g, outs


def time_arms(graphs, per):
    ts = {k: [] for k in graphs}
    for g in graphs.values():
        g.replay()
    torch.cuda.synchronize()
    for _ in range(ROUNDS):
        for k, g in graphs.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            g.replay()
            b.record()
            b.synchronize()
            ts[k].append(a.elapsed_time(b) * 1000.0 / per)
    return {k: round(statistics.median(v), 2) for k, v in ts.items()}


def flat(o):
    return [t for t in (o if isinstance(o, (tuple, list)) else (o,)) if t is not None]


def row(name, make, fn, exact):
    res = {"workload": name}
    for hn, hd in HALVES.items():
        half_sets = make(hd)
        wide_sets = [tuple(t.float() if (t is not None and t.dtype == hd) else t for t in s) for s in half_sets]
        graphs, outs = {}, {}
        graphs["fp32"], outs["fp32"] = graph_of(fn, wide_sets, False)
        graphs[hn], outs[hn] = graph_of(fn, half_sets, False)
        graphs[hn + "+cast"], outs[hn + "+cast"] = graph_of(fn, half_sets, True)
        us = time_arms(graphs, REPS * len(half_sets))
        for k in graphs:
            graphs[k].replay()
        torch.cuda.synchronize()
        ok = True
        for a, b, c in zip(outs["fp32"], outs[hn], outs[hn + "+cast"]):
            for ta, tb, tc in zip(flat(a), flat(b), flat(c)):
                ok = ok and torch.equal(ta, tc)
                if exact:
                    ok = ok and torch.equal(ta, tb)
                else:
                    ok = ok and tb.dtype == hd and float((tb.float() - ta).abs().max()) <= 2e-3
        res[hn] = {"us_per_call": us, "sets": len(half_sets), "outputs_agree": bool(ok)}
        del graphs, outs, half_sets, wide_sets
        torch.cuda.empty_cache()
    print(json.dumps(res), flush=True)
    return res


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    _lib.load()
    info = {"card": card(), "torch": torch.__version__, "reps": REPS, "rounds": ROUNDS,
            "l2_bytes_rotated_past": 2 * L2_BYTES, "unit": "us per call, median of the alternated rounds"}
    print(json.dumps(info), flush=True)
    rows = []
    for frames, (b, f) in ((32, (8, 4)), (128, (32, 4))):
        rows.append(row("corr4d_vgg %d frames" % frames, lambda dt, b=b, f=f: corr_sets(b, f, dt), corr_call, False))
    for L in (1, 8):
        rows.append(row("warp_pack lowres 480x854 L=%d" % L,
                        lambda dt, L=L: warp_sets(L, 1, 480, 854, 256, 256, True, dt), warp_call(True), True))
    for frames, (b, f) in ((32, (8, 4)), (128, (32, 4))):
        rows.append(row("warp dense 256x256 %d frames" % frames,
                        lambda dt, b=b, f=f: warp_sets(b, f, 256, 256, 256, 256, False, dt), warp_call(False), True))
    info["rows"] = rows
    if out_path:
        with open(out_path, "w") as fh:
            json.dump(info, fh, indent=1)


if __name__ == "__main__":
    main()
