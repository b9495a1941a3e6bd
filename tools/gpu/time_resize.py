"""Event-timed resampling of DFPN's training step at BASELINE cfg3 sizes (B = 32, frames_n 5, 256 x 256): the eager
path (oracle/torch_port.py's restatement of TransformsUtils.resize_set / FlowsUtils.resize_flow on CUDA tensors, i.e.
ATen's transposes + F.interpolate + autograd) against the library's kernels (ops.resize_set / ops.resize_flow), the two
alternated call by call in one process.  Two input sets rotate (each set is > 126 MB of L2).  Prints one JSON document:
us per call (median), the kernels' algorithmic bytes and their rate as a share of the copy bandwidth measured in the same
run, the device name and its power limit.

    python tools/gpu/time_resize.py [out.json]
"""
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from master_thesis_b200 import ops                    # noqa: E402
from oracle import torch_port as tp                    # noqa: E402

B, N, HW = 32, 5, 256
T = N // 2
R_LIST = [i for i in range(N) if i != T]
REPS, WARM = 40, 5


def lin_rows(n_in, n_out):
    """Source indices the bilinear taps touch (ATen's source index, align_corners=False)."""
    if n_in == n_out:
        return set(range(n_in))
    sc = torch.tensor(n_in, dtype=torch.float32) / n_out
    s = torch.clamp(sc * (torch.arange(n_out, dtype=torch.float32) + 0.5) - 0.5, min=0)
    i0 = torch.clamp(torch.floor(s).long(), max=n_in - 1)
    return set(i0.tolist()) | set(torch.clamp(i0 + 1, max=n_in - 1).tolist())


def near_rows(n_in, n_out):
    sc = torch.tensor(n_in, dtype=torch.float32) / n_out
    return set(torch.clamp(torch.floor(torch.arange(n_out, dtype=torch.float32) * sc).long(), max=n_in - 1).tolist())


def bytes_resize_set(s, c=3):
    """Whole source rows (a 32-byte sector holds 8 taps' worth of columns) of the tapped rows, plus the outputs."""
    frames = B * N
    rd = (2 * c * len(lin_rows(HW, s)) + len(near_rows(HW, s))) * HW * 4
    return frames * (rd + (2 * c + 1) * s * s * 4)


def bytes_flow_nearest(s):
    return B * len(R_LIST) * (len(near_rows(HW, s)) * HW * 8 + s * s * 8)


def bytes_flow_up(h, H):
    return B * len(R_LIST) * (h * h * 8 + H * H * 8)


def median_pair(eager, kernel, sets):
    """Median event time (us) of each callable over REPS calls, the two alternated; inputs rotate over ``sets``."""
    for i in range(WARM):
        eager(sets[i % len(sets)])
        kernel(sets[i % len(sets)])
    torch.cuda.synchronize()
    te, tk = [], []
    for r in range(REPS):
        for fn, acc in ((eager, te), (kernel, tk)) if r % 2 == 0 else ((kernel, tk), (eager, te)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s = sets[r % len(sets)]
            e0.record()
            fn(s)
            e1.record()
            torch.cuda.synchronize()
            acc.append(e0.elapsed_time(e1) * 1e3)
    te.sort()
    tk.sort()
    return te[len(te) // 2], tk[len(tk) // 2]


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


def power_limit():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                                        str(torch.cuda.current_device())], text=True, timeout=30).strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    if not torch.cuda.is_available():
        raise SystemExit("time_resize.py measures on a CUDA device; none is visible")
    torch.manual_seed(0)
    sets = []
    for _ in range(2):
        x = torch.rand(B, 3, N, HW, HW, device="cuda")
        m = (torch.rand(B, 1, N, HW, HW, device="cuda") > 0.8).float()
        y = torch.rand(B, 3, N, HW, HW, device="cuda")
        flow_gt = torch.rand(B, N, HW, HW, 2, device="cuda") * 2 - 1
        f64 = (torch.rand(B, len(R_LIST), 2, 64, 64, device="cuda") * 2 - 1).permute(0, 1, 3, 4, 2)
        g256 = torch.rand(B, len(R_LIST), 256, 256, 2, device="cuda") - 0.5
        sets.append(dict(x=x, v=1 - m, y=y, fgt=flow_gt[:, R_LIST], f64=f64, g256=g256))
    bw = copy_bandwidth()
    rows = []

    def row(name, eager, kernel, nbytes):
        te, tk = median_pair(eager, kernel, sets)
        rows.append(dict(call=name, eager_us=round(te, 1), kernel_us=round(tk, 1), speedup=round(te / tk, 2),
                         kernel_bytes=nbytes, kernel_GBps=round(nbytes / (tk * 1e-6) / 1e9, 1),
                         kernel_share_of_copy_bw=round(nbytes / (tk * 1e-6) / 1e9 / bw, 3)))
        print(json.dumps(rows[-1]), flush=True)

    with torch.no_grad():
        for s in (16, 64):
            row("resize_set(x, 1 - m, y, %d)" % s, lambda d: tp.resize_set(d["x"], d["v"], d["y"], s),
                lambda d: ops.resize_set(d["x"], d["v"], d["y"], s), bytes_resize_set(s))
        for s in (16, 64):
            row("resize_flow(flow_gt[:, r_list], (%d, %d))" % (s, s), lambda d: tp.resize_flow(d["fgt"], (s, s)),
                lambda d: ops.resize_flow(d["fgt"], (s, s), "nearest"), bytes_flow_nearest(s))
        row("resize_flow(flow_64, (256, 256), 'bilinear') forward",
            lambda d: tp.resize_flow(d["f64"], (256, 256), "bilinear"),
            lambda d: ops.resize_flow(d["f64"], (256, 256), "bilinear"), bytes_flow_up(64, 256))

    def fwd_bwd(fn):
        def run(d):
            f = d["f64"].detach().requires_grad_(True)
            torch.autograd.backward(fn(f, (256, 256), "bilinear"), d["g256"])
        return run
    row("resize_flow(flow_64, (256, 256), 'bilinear') forward + backward", fwd_bwd(tp.resize_flow),
        fwd_bwd(ops.resize_flow), 2 * bytes_flow_up(64, 256))
    doc = dict(device=torch.cuda.get_device_name(), power_limit=power_limit(), copy_GBps=round(bw, 1),
               sizes=dict(B=B, frames_n=N, HW=HW, refs=len(R_LIST)), reps=REPS, rows=rows)
    text = json.dumps(doc, indent=1)
    print(text)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
