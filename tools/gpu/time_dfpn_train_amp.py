"""Mixed-precision DFPN training: the training-step kernels reading half flows / volumes / VGG features natively,
against the fp32 kernels, and against what a user would otherwise write under autocast (an eager ``.float()`` of the
half operand, then the fp32 kernel, then ``.to(dtype)`` of the gradient).

Arms, per workload (cfg3 sizes: B = 32, F = 4 reference frames):
  fp32       fp32 operands (the half operands widened), the fp32 entry points
  <dt>       fp16 / bf16 operands read by the *_dt entry points, under autocast
  <dt>+cast  the same half operands copied to fp32 by an eager cast, the fp32 entry points, gradients cast back
Workloads: warp_masked_l1 forward + backward at 64 x 64 and 256 x 256; corr4d_l1 forward + backward at 32 and 128
frames; the resize_flow backward 16 -> 64 and 64 -> 256; the whole patched DFPN.compute_loss forward + backward.

The kernel workloads are one CUDA graph of REPS passes over K input sets whose total size exceeds twice the 126 MB
L2, so each pass reads its operands from HBM; CUDA events around graph replays, the arms alternate ROUNDS times, the
median per arm is reported.  The compute_loss workload runs eagerly (autograd), timed the same way around STEPS
steps; its frames alone (2 x 126 MB) exceed the L2.  Outputs are compared in the same run: the warp and resize arms
bit for bit (<dt> against <dt>+cast); the correlation loss of <dt> against fp32 within 2e-3 relative (the fp32 arm
runs kind::tf32, the half arm kind::f16) and <dt>+cast against fp32 bit for bit.

    python tools/gpu/time_dfpn_train_amp.py [out.json]
"""
import json
import os
import statistics
import subprocess
import sys
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from master_thesis_b200 import _lib, ops, plug    # noqa: E402

L2_BYTES = 126 * 2 ** 20
REPS = 4
ROUNDS = 7
STEPS = 5
B, F = 32, 4
HALVES = {"fp16": torch.float16, "bf16": torch.bfloat16}


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


def flow_of(g, b, f, h, w, dt, sigma=0.03):
    base = torch.stack(torch.meshgrid(torch.linspace(-1, 1, h, device="cuda"), torch.linspace(-1, 1, w, device="cuda"),
                                      indexing="ij")[::-1], -1)
    return (base + sigma * torch.randn((b, f, h, w, 2), device="cuda", generator=g)).to(dt)


# ---------------------------------------------------------------- workloads: (make(dt) -> sets, call(set, dt, cast))
def warp_l1_sets(size):
    def make(dt):
        g = torch.Generator(device="cuda").manual_seed(size)
        one = B * (F + 1) * 4 * size * size * 4 + B * F * size * size * 2 * 4
        sets = []
        for _ in range(n_sets(one)):
            x = torch.rand((B, 3, F + 1, size, size), device="cuda", generator=g)
            v = (torch.rand((B, 1, F + 1, size, size), device="cuda", generator=g) > 0.1).float()
            sets.append((x[:, :, 1:], v[:, :, 1:], flow_of(g, B, F, size, size, dt), x[:, :, 0], v[:, :, 0]))
        return sets
    return make


def warp_l1_call(s, dt, cast):
    x, v, flow, xt, vt = s
    if cast:
        flow = flow.float()
    out3, _, _, saved = ops.warp_l1_fwd_raw(x, v, flow, xt, vt)
    g = ops.warp_l1_bwd_raw(saved, out3[:1])
    return out3, (g.to(dt) if cast else g)


def corr_l1_sets(b, f):
    def make(dt):
        g = torch.Generator(device="cuda").manual_seed(b * 10 + f)
        one = b * 512 * (f + 1) * 256 * 2 + b * f * 65536 * 3
        sets = []
        for _ in range(n_sets(one)):
            ft = torch.relu(torch.randn((b, 512, 16, 16), device="cuda", generator=g)).to(dt)
            fr = torch.relu(torch.randn((b, 512, f, 16, 16), device="cuda", generator=g)).to(dt)
            pred = torch.rand((b, f, 16, 16, 16, 16), device="cuda", generator=g).to(dt)
            sets.append((pred, ft, fr))
        return sets
    return make


def corr_l1_call(s, dt, cast):
    pred, ft, fr = s
    if cast:
        pred, ft, fr = pred.float(), ft.float(), fr.float()
    loss, sign = ops.corr4d_l1_fwd_raw(pred, ft, fr)
    gp = ops.Corr4dL1Fn.backward(types.SimpleNamespace(sign=sign, dtype=pred.dtype), loss)[0]
    return loss, (gp.to(dt) if cast else gp)


def resize_bwd_sets(h, H):
    def make(dt):
        g = torch.Generator(device="cuda").manual_seed(h)
        one = B * F * H * H * 2 * 4 + B * F * h * h * 2 * 4
        return [(torch.randn((B, F, H, H, 2), device="cuda", generator=g), torch.empty(0, dtype=dt, device="cuda"))
                for _ in range(n_sets(one))]
    return make


def resize_bwd_call(h):
    def call(s, dt, cast):
        gout, like = s
        if cast or like.dtype == torch.float32:
            gf = ops.resize_flow_bwd_raw(gout, h, h)
            return (gf.to(dt) if cast else gf,)
        return (ops.resize_flow_bwd_raw(gout, h, h, like.dtype),)
    return call


# ---------------------------------------------------------------- timing
def graph_of(call, sets, dt, cast):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s), torch.autocast("cuda", dtype=dt):
        for st in sets:           # warm-up: module load, tensor maps, allocator
            call(st, dt, cast)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g), torch.autocast("cuda", dtype=dt):
        for _ in range(REPS):
            outs = [call(st, dt, cast) for st in sets]
    return g, outs


def time_arms(runs, per):
    ts = {k: [] for k in runs}
    for r in runs.values():
        r()
    torch.cuda.synchronize()
    for _ in range(ROUNDS):
        for k, r in runs.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            r()
            b.record()
            b.synchronize()
            ts[k].append(a.elapsed_time(b) * 1000.0 / per)
    return {k: round(statistics.median(v), 2) for k, v in ts.items()}


def kernel_row(name, make, call, loss_rtol=None):
    res = {"workload": name}
    for hn, hd in HALVES.items():
        try:
            half_sets = make(hd)
            wide_sets = [tuple(t.float() if t.dtype == hd else t for t in s) for s in half_sets]
            graphs, outs = {}, {}
            graphs["fp32"], outs["fp32"] = graph_of(call, wide_sets, hd, False)
            graphs[hn], outs[hn] = graph_of(call, half_sets, hd, False)
            graphs[hn + "+cast"], outs[hn + "+cast"] = graph_of(call, half_sets, hd, True)
            us = time_arms({k: g.replay for k, g in graphs.items()}, REPS * len(half_sets))
            for g in graphs.values():
                g.replay()
            torch.cuda.synchronize()
            ok = True
            for a, b, c in zip(outs["fp32"], outs[hn], outs[hn + "+cast"]):
                ok = ok and torch.equal(a[0].to(c[0].dtype), c[0])  # the cast arm: the fp32 kernel on the same values
                ok = ok and b[-1].dtype == hd and c[-1].dtype == hd
                if loss_rtol is None:
                    ok = ok and all(torch.equal(tb, tc) for tb, tc in zip(b, c))
                else:
                    ok = ok and abs(float(b[0]) - float(a[0])) <= loss_rtol * abs(float(a[0]))
            res[hn] = {"us_per_call": us, "sets": len(half_sets), "outputs_agree": bool(ok)}
            del graphs, outs, half_sets, wide_sets
        except Exception as e:      # one failing arm does not hide the others' numbers
            res[hn] = {"error": "%s: %s" % (type(e).__name__, e)}
        torch.cuda.empty_cache()
    print(json.dumps(res), flush=True)
    return res


class _Nets(object):
    """The DFPN stand-in of step_row: its forward returns the leaves, its VGG constant features; ``cast``: both are
    handed over as eager fp32 copies."""

    def __init__(self, nets, feats, cast):
        self.nets, self.feats, self.cast = nets, feats, cast

    def __call__(self, *a):
        return tuple(v.float() for v in self.nets) if self.cast else tuple(self.nets)

    def model_vgg(self, inp):
        return [None, None, None, self.feats.float() if self.cast else self.feats]


def step_row():
    """The patched DFPN._train_val_wrapper + DFPN.compute_loss forward + backward at cfg3 sizes (256 x 256, B = 32,
    F = 4) with stand-ins for the networks: corr / flows as leaves, constant VGG features."""
    res = {"workload": "patched compute_loss fwd+bwd 256x256 B=32 F=4"}
    stub = types.ModuleType("master_thesis")
    stub.TransformsUtils = types.SimpleNamespace(resize_set=plug.TransformsUtils.resize_set)
    stub.FlowsUtils = types.SimpleNamespace(resize_flow=plug.FlowsUtils.resize_flow)
    saved = sys.modules.get("master_thesis")
    sys.modules["master_thesis"] = stub
    try:
        n, t = F + 1, (F + 1) // 2
        r_list = [i for i in range(n) if i != t]
        g = torch.Generator(device="cuda").manual_seed(7)
        x = torch.rand((B, 3, n, 256, 256), device="cuda", generator=g)
        m = (torch.rand((B, 1, n, 256, 256), device="cuda", generator=g) < 0.1).float()
        y = torch.rand((B, 3, n, 256, 256), device="cuda", generator=g)
        flow_gt = flow_of(g, B, n, 256, 256, torch.float32)
        use = torch.ones(B, dtype=torch.bool, device="cuda")
        nets32 = [torch.rand((B, F, 16, 16, 16, 16), device="cuda", generator=g)] + \
            [flow_of(g, B, F, s, s, torch.float32) for s in (16, 64, 256)]
        feats32 = torch.relu(torch.randn((B * n, 512, 16, 16), device="cuda", generator=g))
        for hn, hd in HALVES.items():
            try:
                arms = {"fp32": (torch.float32, False), hn: (hd, False), hn + "+cast": (hd, True)}
                losses, runs = {}, {}
                for arm, (dt, cast) in arms.items():
                    nets = [a.to(dt).requires_grad_(True) for a in nets32]

                    def step(fake=_Nets(nets, feats32.to(dt), cast), nets=nets, dt=dt, arm=arm):
                        with torch.autocast("cuda", dtype=hd, enabled=dt != torch.float32):
                            r = plug.dfpn_train_val_wrapper(fake, x, m, y, flow_gt, use, t, r_list)
                            loss, _ = plug.dfpn_compute_loss(fake, *r, t, r_list)
                        grads = torch.autograd.grad(loss, nets)
                        losses[arm] = (loss.detach(), grads)

                    runs[arm] = lambda step=step: [step() for _ in range(STEPS)]
                us = time_arms(runs, STEPS)
                l32, lh, lc = float(losses["fp32"][0]), float(losses[hn][0]), float(losses[hn + "+cast"][0])
                ok = abs(lh - lc) <= 2e-3 * abs(lc) and all(gr.dtype == hd for gr in losses[hn][1])
                res[hn] = {"us_per_step": us, "loss": {"fp32": l32, hn: lh, hn + "+cast": lc}, "outputs_agree": bool(ok)}
            except Exception as e:
                res[hn] = {"error": "%s: %s" % (type(e).__name__, e)}
            torch.cuda.empty_cache()
    finally:
        if saved is None:
            del sys.modules["master_thesis"]
        else:
            sys.modules["master_thesis"] = saved
    print(json.dumps(res), flush=True)
    return res


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    _lib.load()
    info = {"card": card(), "torch": torch.__version__, "reps": REPS, "rounds": ROUNDS, "steps": STEPS,
            "l2_bytes_rotated_past": 2 * L2_BYTES, "unit": "us per call (per step), median of the alternated rounds"}
    print(json.dumps(info), flush=True)
    rows = []
    for size in (64, 256):
        rows.append(kernel_row("warp_masked_l1 fwd+bwd %dx%d B=%d F=%d" % (size, size, B, F), warp_l1_sets(size),
                               warp_l1_call))
    for frames, (b, f) in ((32, (8, 4)), (128, (32, 4))):
        rows.append(kernel_row("corr4d_l1 fwd+bwd %d frames" % frames, corr_l1_sets(b, f), corr_l1_call, 2e-3))
    for h, H in ((16, 64), (64, 256)):
        rows.append(kernel_row("resize_flow bwd %d->%d B=%d F=%d" % (h, H, B, F), resize_bwd_sets(h, H),
                               resize_bwd_call(h)))
    rows.append(step_row())
    info["rows"] = rows
    if out_path:
        with open(out_path, "w") as fh:
            json.dump(info, fh, indent=1)


if __name__ == "__main__":
    main()
