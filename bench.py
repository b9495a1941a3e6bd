#!/usr/bin/env python
"""bench.py - aligned frames/s of the frame-alignment hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg2] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input.  The
default workload ("align") is the north_star's "DFPN+CPN alignment of 5-frame
256x256 clips", batch_size=8: BASELINE.json configs[1] (cfg2: the CPN.align tail
- affine warp + visibility + v_maps, model_cpn.py:75-89 - on 32 (b, ref) frames
followed by CM_Module, model_cpn.py:206-254) PLUS the DFPN aligner's hot path on
the same batch (correlation_masked_4d on tcgen05, model_dfpn.py:534-565, and the
DFPN.align tail, model_dfpn.py:128-133), so that the one line carries both halves
of the metric: an HBM roofline (`roofline`) and a tensor-core one (`roofline_tc`).
--workload cfg1..cfg5 time the individual configs' hot paths; see WORKLOADS.

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for the meaning
of every key.  N > 1: launched under torchrun (one rank per GPU); the batch is
sharded by sample, every rank runs the same per-GPU batch (weak scaling), no
data-path collective.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


OUT = None


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), float(p["bf16_tflops"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------
# workloads
# ---------------------------------------------------------------------------
CORR_FLOP = 2 * 256 * 256 * 512     # per (b, f) frame: M = N = 256, K = 512 (SURVEY 8d: 67.1 MFLOP)

class Workload(object):
    """Synthetic inputs + one hot-path step.  ``calls`` names the C-ABI calls of a
    step in order with their algorithmic bytes (SURVEY.md 8d) and kernel launches."""
    name = ""
    describe = ""
    frames_per_step = 0

    def host_inputs(self, seed):
        raise NotImplementedError

    def gpu_step(self, mtb, d):
        raise NotImplementedError

    def cpu_step(self, tp, d):
        raise NotImplementedError

    def calls(self):
        raise NotImplementedError


class Cfg2(Workload):
    """CPN alignment tail + context matching, B=8, frames_n=5, 256x256."""
    name = "cfg2"

    def __init__(self, b=8, f=4, h=256, w=256, c=128):
        self.b, self.f, self.h, self.w, self.c = b, f, h, w, c
        self.frames_per_step = b * f
        self.describe = ("cfg2: CPN.align tail (affine warp+visibility+v_maps) + CM_Module, "
                         "batch_size=%d frames_n=%d %dx%d c_feats=%dx%dx%d per GPU"
                         % (b, f + 1, h, w, c, h // 4, w // 4))

    def host_inputs(self, seed):
        import numpy as np
        from master_thesis_b200 import synth
        b, f, h, w, c = self.b, self.f, self.h, self.w, self.c
        x, m, _ = synth.frames(seed, b, f + 1, h, w)
        t = (f + 1) // 2                                    # model_dfpn.py:471-473
        refs = [i for i in range(f + 1) if i != t]
        r = synth.rng(seed + 3)
        return {
            "x_refs": np.ascontiguousarray(x[:, :, refs]),
            "m_refs": np.ascontiguousarray(m[:, :, refs]),
            "m_target": np.ascontiguousarray(m[:, :, t]),
            "v_target": np.ascontiguousarray(1 - m[:, :, t]),
            "theta": synth.thetas(seed + 1, b * f, float(os.environ.get("MT_BENCH_THETA_SIGMA", "0.1"))),
            "c_feats": r.standard_normal((b, c, f + 1, h // 4, w // 4)).astype(np.float32),
        }

    inputs_h2d = ("x_refs", "m_refs", "m_target", "v_target", "theta", "c_feats")

    def gpu_step(self, mtb, d):
        xa, va, vm = mtb.cpn_align_tail(d["x_refs"], d["m_refs"], d["m_target"], d["theta"])
        out, cmask = mtb.ops.cm_match(d["c_feats"], d["v_target"], va)
        return {"x_aligned": xa, "v_aligned": va, "v_maps": vm, "cm_out": out, "c_mask": cmask}

    def cpu_step(self, tp, d):
        xa, va, vm = tp.cpn_align_tail(d["x_refs"], d["m_refs"], d["m_target"], d["theta"])
        out, cmask = tp.cm_module(d["c_feats"], d["v_target"], va)
        return xa, va, vm, out, cmask

    def calls(self):
        px = self.h * self.w
        n = self.b * self.f
        p = (self.h // 4) * (self.w // 4)
        # a3 with in-kernel affine grid: 36*px + 4*px/F per frame (SURVEY 8d: 44px+4px/F minus the 8px grid)
        warp = n * 36 * px + self.b * 4 * px
        # a8 per sample: c_feats + full-res masks in; (2C+1)*P + P out
        cm = self.b * (self.c * (self.f + 1) * p * 4 + (self.f + 1) * px * 4
                       + (2 * self.c + 1) * p * 4 + p * 4)
        return [("mt_warp_fwd", 1, warp, "hbm"), ("mt_cm_match_fwd", 3, cm, "hbm")]

    def sub(self, b):
        return Cfg2(b, self.f, self.h, self.w, self.c)


class Align(Workload):
    """DFPN + CPN alignment of 5-frame 256x256 clips (north_star): both aligners' hot paths on the same
    batch - DFPN: masked VGG correlation (tcgen05) + flow warp / visibility / v_map; CPN: affine warp /
    visibility / v_map (BASELINE configs[1]) + context matching."""
    name = "align"

    def __init__(self, b=8, f=4, h=256, w=256, c=128):
        self.b, self.f, self.h, self.w, self.c = b, f, h, w, c
        self.cpn, self.dfpn = Cfg2(b, f, h, w, c), Cfg1(b, f, h, w)
        self.frames_per_step = 2 * b * f
        self.describe = ("align: DFPN+CPN alignment hot paths, batch_size=%d frames_n=%d %dx%d per GPU = %d aligned "
                         "frames per step (%d per aligner): correlation_masked_4d 512x16x16 (tcgen05) + DFPN.align "
                         "tail | CPN.align tail (BASELINE configs[1]) + CM_Module on c_feats %dx%dx%d"
                         % (b, f + 1, h, w, 2 * b * f, b * f, c, h // 4, w // 4))

    def host_inputs(self, seed):
        d = self.cpn.host_inputs(seed)
        d.update({k: v for k, v in self.dfpn.host_inputs(seed).items() if k not in d})
        return d

    def gpu_step(self, mtb, d):
        # one stream: capturing the two aligners' paths as parallel graph branches was measured (r2, call M: 104.5 vs
        # 102.0 us) - every kernel here is a persistent one-CTA-per-SM kernel with ~200 KB of shared memory, so two
        # of them never share an SM and the branches only interleave
        out = self.dfpn.gpu_step(mtb, d)
        out.update({"cpn_" + k: v for k, v in self.cpn.gpu_step(mtb, d).items()})
        return out

    def cpu_step(self, tp, d):
        return self.dfpn.cpu_step(tp, d) + self.cpn.cpu_step(tp, d)

    def calls(self):
        return self.dfpn.calls() + self.cpn.calls()

    def sub(self, b):
        return Align(b, self.f, self.h, self.w, self.c)


class Cfg1(Workload):
    """DFPN alignment hot path: masked correlation + flow warp, B=8, frames_n=2, 256x256."""
    name = "cfg1"

    def __init__(self, b=8, f=1, h=256, w=256):
        self.b, self.f, self.h, self.w = b, f, h, w
        self.frames_per_step = b * f
        self.describe = ("cfg1: DFPN hot path (correlation_masked_4d 512x16x16 + align tail), "
                         "batch_size=%d frames_n=%d %dx%d per GPU" % (b, f + 1, h, w))

    def host_inputs(self, seed):
        import numpy as np
        from master_thesis_b200 import synth
        b, f, h, w = self.b, self.f, self.h, self.w
        x, m, _ = synth.frames(seed, b, f + 1, h, w)
        t = (f + 1) // 2
        refs = [i for i in range(f + 1) if i != t]
        ft, vt, fr, vr = synth.vgg_feats(seed + 2, b, f)
        return {
            "x_refs": np.ascontiguousarray(x[:, :, refs]),
            "m_refs": np.ascontiguousarray(m[:, :, refs]),
            "m_target": np.ascontiguousarray(m[:, :, t]),
            "flow": synth.dense_flow(seed + 1, b, f, h, w, 0.05, True),
            "feats_t": ft, "v_t16": vt, "feats_r": fr, "v_r16": vr,
        }

    inputs_h2d = ("x_refs", "m_refs", "m_target", "flow", "feats_t", "v_t16", "feats_r", "v_r16")

    def gpu_step(self, mtb, d):
        corr = mtb.ops.corr4d(d["feats_t"], d["v_t16"], d["feats_r"], d["v_r16"])
        xa, va, vm = mtb.dfpn_align_tail(d["x_refs"], d["m_refs"], d["m_target"], d["flow"])
        return {"corr": corr, "x_aligned": xa, "v_aligned": va, "v_maps": vm}

    def cpu_step(self, tp, d):
        corr = tp.corr4d(d["feats_t"], d["v_t16"], d["feats_r"], d["v_r16"])
        return (corr,) + tuple(tp.dfpn_align_tail(d["x_refs"], d["m_refs"], d["m_target"], d["flow"]))

    def calls(self):
        px = self.h * self.w
        n = self.b * self.f
        warp = n * 44 * px + self.b * 4 * px
        corr = n * (524288 + 262144) + self.b * 524288 + (n + self.b) * 1024
        return [("mt_corr4d_fwd", 1, corr, "tensor", n * CORR_FLOP), ("mt_warp_fwd", 1, warp, "hbm")]

    def sub(self, b):
        return Cfg1(b, self.f, self.h, self.w)


class Cfg4(Workload):
    """CHN inference hot path with the DFPN aligner on one DAVIS-shaped frame pair."""
    name = "cfg4"

    def __init__(self, b=1, f=1, h=480, w=854):
        self.b, self.f, self.h, self.w = b, f, h, w
        self.frames_per_step = b * f
        self.describe = ("cfg4: CHN inference hot path, DFPN aligner (warp + pack | composite + "
                         "hole update: two kernels), batch_size=%d F=%d %dx%d per GPU" % (b, f, h, w))

    def host_inputs(self, seed):
        import numpy as np
        from master_thesis_b200 import synth
        b, f, h, w = self.b, self.f, self.h, self.w
        x, m, _ = synth.frames(seed, b, f + 1, h, w)
        return {
            "x_target": np.ascontiguousarray(x[:, :, 0]),
            "x_refs": np.ascontiguousarray(x[:, :, 1:]),
            "m_refs": np.ascontiguousarray(m[:, :, 1:]),
            "m_target": np.ascontiguousarray(m[:, :, 0]),
            "v_target": np.ascontiguousarray(1 - m[:, :, 0]),
            "flow": synth.dense_flow(seed + 1, b, f, h, w, 0.03, True),
            "nn_out": synth.nn_output(seed + 2, b * f, h, w),
        }

    inputs_h2d = ("x_target", "x_refs", "m_refs", "m_target", "v_target", "flow", "nn_out")

    def gpu_step(self, mtb, d):
        # the step of CHN.inpaint_* as the patched loop runs it (plug._fill_step): warp + CNN-input pack in
        # one kernel, [RRDBNet: cuDNN, outside the hot path], composite + hole update in one kernel
        ops = mtb.ops
        nn_in, vm, _, _ = ops.warp_pack_fwd(d["x_refs"], d["m_refs"], d["flow"], d["m_target"], d["x_target"],
                                            d["v_target"], ops.ALIGN_CORNERS | ops.VIS_FROM_MASK)
        y_comp, m_new, x_new, per = ops.chn_fill(d["nn_out"], d["x_target"], d["v_target"], d["m_target"],
                                                 vm[:, :, 0])
        return {"nn_in": nn_in, "y_comp": y_comp, "m_new": m_new, "x_new": x_new, "inp_per": per}

    def cpu_step(self, tp, d):
        xa, va, vm = tp.dfpn_align_tail(d["x_refs"], d["m_refs"], d["m_target"], d["flow"])
        nn_in = tp.chn_pack(d["x_target"], d["v_target"], xa, va, vm)
        y_hat, y_comp = tp.chn_composite(d["nn_out"], d["x_target"], d["v_target"], self.b, self.f)
        return nn_in, tp.hole_update(d["m_target"], vm[:, :, 0], y_comp[:, :, 0])

    def calls(self):
        px = self.h * self.w
        n = self.b * self.f
        # warp + pack: x_ref 12, m_ref 4, flow 8 in; nn_in 36, v_map 4 out; per sample x_t 12, v_t 4, m_t 4 in
        # composite + hole update (F = 1): nn_out 12, x_t 12, v_t 4, m_t 4, v_map 4 in; y_comp 12, m_new 4, x_new 12 out
        return [("mt_warp_pack_fwd", 1, n * 64 * px + self.b * 20 * px, "hbm"),
                ("mt_chn_fill_step", 1, self.b * 64 * px, "hbm")]

    def sub(self, b):
        return Cfg4(b, self.f, self.h, self.w)

    def loop_stats(self, mtb, dev, n=8, reps=3):
        """Loop level (SURVEY 8f-4): the patched CHN.inpaint_ff over an n-frame 480x854 clip with stand-ins for the two
        CNNs (the DFPN forward hands out a 256x256 flow, the RRDBNet a preset tensor - both outside the hot path), timed
        with one device->host sync per step (the reference's loop control, model_chn.py:112) and with the loop condition
        evaluated on the device and the host looking every 8 steps."""
        import time
        import numpy as np
        import torch
        from master_thesis_b200 import plug, synth
        h, w = self.h, self.w
        x, m, _ = synth.frames(77, 1, n, h, w)
        x, m = torch.from_numpy(x[0]).to(dev), torch.from_numpy(m[0]).to(dev)          # (3, n, H, W), (1, n, H, W)
        flow = torch.from_numpy(synth.dense_flow(78, 1, 1, 256, 256, 0.03, True)).to(dev)
        nn_o = torch.from_numpy(synth.nn_output(79, 1, h, w)).to(dev)
        steps = [0]

        class _DFPN(object):
            align = plug.dfpn_align

            def __call__(self, *a):
                return None, None, None, flow

        class _CHN(object):
            forward = plug.chn_forward
            inpaint_ff = plug.chn_inpaint_ff
            model_aligner = _DFPN()

            @staticmethod
            def get_indexes_ff(t, n_frames, s=1, D=20):
                return sorted((i for i in range(n_frames) if i != t), key=lambda i: abs(i - t))[:D]

            def nn(self, inp):
                steps[0] += 1
                return nn_o

            def __call__(self, *a):
                return self.forward(*a)

        out = {}
        for k in (1, 8):
            chn = _CHN()
            chn.mt_b200_sync_every = k
            chn.inpaint_ff(x, m)                      # warm-up
            torch.cuda.synchronize()
            steps[0] = 0
            t0 = time.perf_counter()
            for _ in range(reps):
                y = chn.inpaint_ff(x, m)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            out["sync_every_%d" % k] = {"target_frames_per_sec": reps * n / dt, "fill_steps_per_target": steps[0] / (reps * n),
                                        "us_per_fill_step": 1e6 * dt / max(steps[0], 1)}
        out["note"] = ("patched CHN.inpaint_ff on an %d-frame %dx%d clip, host-driven loop (Python + 2 C-ABI calls per fill step), "
                       "CNN stand-ins; the kernel-level step above is %s" % (n, h, w, "the two kernels alone"))
        return out


class Cfg3(Workload):
    """DFPN training-step hot path as the patched reference runs it: the masked correlation of the forward
    pass (CorrelationVGG.forward -> correlation_masked_4d, model_dfpn.py:528) and the patched
    DFPN.compute_loss (plug.dfpn_compute_loss, model_dfpn.py:210-293) with its backward: unmasked correlation
    of the ground truth, three flow L1 losses, and the fused warp + mask_out + masked-L1 reconstruction terms
    at the 64 and 256 scales (forward, and one backward kernel each that writes only d loss / d flow)."""
    name = "cfg3"
    graph_ok = False     # the recorded step also runs the reference's own eager ops; only the kernels are replayed

    def __init__(self, b=32, f=4, h=256, w=256):
        self.b, self.f, self.h, self.w = b, f, h, w
        self.frames_per_step = b * f
        self.describe = ("cfg3: DFPN training hot path through the patched DFPN.compute_loss (2x "
                         "correlation_masked_4d 512x16x16 - the second with F.l1_loss(corr, corr_y) in its epilogue, fwd/bwd -, 3 flow-L1 fwd/bwd, fused warp+mask_out+masked-L1 fwd/bwd "
                         "at %dx%d and %dx%d), batch_size=%d frames_n=%d per GPU" % (h, w, h // 4, w // 4, b, f + 1))

    def host_inputs(self, seed):
        import numpy as np
        from master_thesis_b200 import synth
        b, f, h, w = self.b, self.f, self.h, self.w
        r = synth.rng(seed + 9)
        d = {"flows_use": (r.random_sample(b) < 0.75).astype(np.float32),
             "corr_in": r.random_sample((b, f, 16, 16, 16, 16)).astype(np.float32)}
        for tag, (hh, ww) in (("", (h, w)), ("_s", (h // 4, w // 4)), ("_t", (16, 16))):
            x, m, y = synth.frames(seed + len(tag), b, f + 1, hh, ww)
            d["x" + tag], d["v" + tag] = x, 1 - m
            d["flow" + tag] = synth.dense_flow(seed + 1, b, f, hh, ww, 0.05, True)
            d["flow_gt" + tag] = synth.dense_flow(seed + 2, b, f, hh, ww, 0.05, True)
        ft, vt, fr, vr = synth.vgg_feats(seed + 2, b, f)
        d.update({"feats_t": ft, "v_t16": vt, "feats_r": fr, "v_r16": vr,
                  "feats_y": np.maximum(r.standard_normal((b * (f + 1), 512, 16, 16)), 0).astype(np.float32)})
        return d

    def gpu_step(self, mtb, d):
        import torch
        plug = mtb.plug
        f = self.f
        t = (f + 1) // 2
        r_list = [i for i in range(f + 1) if i != t]
        out = {"corr": plug.CorrelationVGG.correlation_masked_4d(d["feats_t"], d["v_t16"], d["feats_r"], d["v_r16"])}
        flows = tuple(d["flow" + tag].detach().requires_grad_(True) for tag in ("_t", "_s", ""))
        flows_gt = tuple(d["flow_gt" + tag] for tag in ("_t", "_s", ""))
        xs = tuple(d["x" + tag] for tag in ("_t", "_s", ""))
        vs = tuple(d["v" + tag] for tag in ("_t", "_s", ""))
        xs_aligned = tuple(plug.DeferredAlign(x[:, :, r_list], v[:, :, r_list], fl) for x, v, fl in zip(xs, vs, flows))
        corr_in = d["corr_in"].detach().requires_grad_(True)
        feats_y = d["feats_y"]

        class _Self(object):               # the two members of the DFPN module compute_loss touches
            @staticmethod
            def model_vgg(inp):
                return [None, None, None, feats_y]

        loss, items = plug.dfpn_compute_loss(_Self(), corr_in, xs, vs, xs, xs_aligned, flows, flows_gt,
                                             d["flows_use"] > 0.5, t, r_list)
        grads = torch.autograd.grad(loss, (corr_in,) + flows)
        out.update({"loss": loss.detach(), "items": torch.stack([i.detach() for i in items]),
                    "g_flow_t": grads[1], "g_flow_s": grads[2], "g_flow": grads[3]})
        return out

    def cpu_step(self, tp, d):
        import torch
        f = self.f
        t = (f + 1) // 2
        r_list = [i for i in range(f + 1) if i != t]
        res = [tp.corr4d(d["feats_t"], d["v_t16"], d["feats_r"], d["v_r16"])]
        flows = tuple(d["flow" + tag].detach().requires_grad_(True) for tag in ("_t", "_s", ""))
        flows_gt = tuple(d["flow_gt" + tag] for tag in ("_t", "_s", ""))
        xs = tuple(d["x" + tag] for tag in ("_t", "_s", ""))
        vs = tuple(d["v" + tag] for tag in ("_t", "_s", ""))
        xs_aligned = tuple(tp.align_set(x[:, :, r_list], v[:, :, r_list], fl)[0] for x, v, fl in zip(xs, vs, flows))
        corr_in = d["corr_in"].detach().requires_grad_(True)
        loss, _ = tp.dfpn_compute_loss(lambda inp: [None, None, None, d["feats_y"]], corr_in, xs, vs, xs, xs_aligned,
                                       flows, flows_gt, d["flows_use"] > 0.5, t, r_list)
        return res + list(torch.autograd.grad(loss, (corr_in,) + flows))

    def calls(self, plan=None):
        """Algorithmic bytes per recorded launch, from the launch's own shape arguments (the order of the
        backward launches is autograd's)."""
        if plan is None:
            raise RuntimeError("cfg3 needs the recorded plan")
        out = []
        for i, name in enumerate(plan.names()):
            a = plan.args(i)
            if name == "mt_corr4d_fwd":
                n = a["B"] * a["F"]
                masks = (n + a["B"]) * 1024 if a["v_t"] else 0
                out.append((name, 1, n * (524288 + 262144) + a["B"] * 524288 + masks, "tensor", n * CORR_FLOP))
            elif name == "mt_corr4d_vgg_l1_fwd":
                # features once, the prediction read (4 B) and the signs written (1 B) per volume element; no volume
                n, pp = a["B"] * a["F"], (a["h"] * a["w"]) ** 2
                out.append((name, 1, n * 524288 + a["B"] * 524288 + n * pp * 5, "tensor", n * CORR_FLOP))
            elif name == "mt_corr4d_l1_bwd":
                out.append((name, 1, a["n"] * 5, "hbm"))             # signs read, gradient written
            elif name in ("mt_warp_l1_fwd", "mt_warp_l1_bwd"):
                n, px = a["B"] * a["F"], a["H"] * a["W"]
                # loss-only fused forward: x_ref 12 + flow 8 per frame, target 12 + v 4 per sample; backward + 8 written
                out.append((name, 1, n * (20 if name.endswith("fwd") else 28) * px + a["B"] * 16 * px, "hbm"))
            elif name in ("mt_masked_l1_fwd", "mt_masked_l1_bwd"):
                el = a["B"] * a["C"] * a["F"] * a["P"]
                out.append((name, 1, el * (8 if name.endswith("fwd") else 12), "hbm"))   # y_hat, y (+ grad written)
            else:
                raise RuntimeError("unexpected launch in the cfg3 step: %s" % name)
        return out

    def sub(self, b):
        return Cfg3(b, self.f, self.h, self.w)


class Cfg5(Workload):
    """CHN training-step hot path with the CPN aligner (model_chn.py:256-280, 324-362): affine warp,
    CNN-input pack, composite, the three masked-L1 terms, and their backward down to the CNN output."""
    name = "cfg5"

    def __init__(self, b=8, f=4, h=256, w=256):
        self.b, self.f, self.h, self.w = b, f, h, w
        self.frames_per_step = b * f
        self.describe = ("cfg5: CHN training hot path, CPN aligner (affine warp + pack + composite "
                         "fwd/bwd + the three masked-L1 terms fwd/bwd in one pass each), batch_size=%d per GPU (64 global on 8 GPUs) "
                         "frames_n=%d %dx%d" % (b, f + 1, h, w))

    def host_inputs(self, seed):
        import numpy as np
        from master_thesis_b200 import synth
        b, f, h, w = self.b, self.f, self.h, self.w
        x, m, y = synth.frames(seed, b, f + 1, h, w)
        t = (f + 1) // 2
        refs = [i for i in range(f + 1) if i != t]
        return {
            "x_target": np.ascontiguousarray(x[:, :, t]), "y_target": np.ascontiguousarray(y[:, :, t]),
            "m_target": np.ascontiguousarray(m[:, :, t]), "v_target": np.ascontiguousarray(1 - m[:, :, t]),
            "x_refs": np.ascontiguousarray(x[:, :, refs]), "m_refs": np.ascontiguousarray(m[:, :, refs]),
            "theta": synth.thetas(seed + 1, b * f, 0.1), "nn_out": synth.nn_output(seed + 2, b * f, h, w),
            "grad_out3": np.ones(3, np.float32),
        }

    def gpu_step(self, mtb, d):
        ops = mtb.ops
        b, f = self.b, self.f
        xa, va, vm = mtb.cpn_align_tail(d["x_refs"], d["m_refs"], d["m_target"], d["theta"])
        nn_in = ops.chn_pack(d["x_target"], d["v_target"], xa, va, vm)
        y_hat, y_comp = ops.chn_composite(d["nn_out"], d["x_target"], d["v_target"], b, f)
        # compute_loss (model_chn.py:347-362): the three masked-L1 terms in one pass, and their autograd
        out9, saved = ops.chn_l1x3_fwd_raw(y_hat, y_comp, d["y_target"], d["v_target"], vm, (0.5, 2.0, 1.0))
        g_yh, g_yc = ops.chn_l1x3_bwd_raw(saved, d["grad_out3"])
        g_nn = ops.chn_composite_bwd_raw(d["nn_out"], d["v_target"], g_yh, g_yc, b, f)
        return {"nn_in": nn_in, "losses": out9, "g_nn": g_nn, "keep": (xa, va, vm, y_hat, y_comp, g_yh, g_yc)}

    def cpu_step(self, tp, d):
        import torch
        b, f = self.b, self.f
        xa, va, vm = tp.cpn_align_tail(d["x_refs"], d["m_refs"], d["m_target"], d["theta"])
        nn_in = tp.chn_pack(d["x_target"], d["v_target"], xa, va, vm)
        nn_out = d["nn_out"].detach().requires_grad_(True)
        y_hat, y_comp = tp.chn_composite(nn_out, d["x_target"], d["v_target"], b, f)
        tgt = d["y_target"].unsqueeze(2).repeat(1, 1, f, 1, 1)
        nh = d["v_target"].unsqueeze(2).repeat(1, 1, f, 1, 1)
        loss = tp.masked_l1(y_hat, tgt, nh, reduction='sum', weight=0.5) + \
            tp.masked_l1(y_hat, tgt, vm, reduction='sum', weight=2) + \
            tp.masked_l1(y_comp, tgt, (1 - nh) - vm, reduction='sum', weight=1)
        return nn_in, torch.autograd.grad(loss, nn_out)[0]

    def calls(self):
        px = self.h * self.w
        n = self.b * self.f
        l1f = n * 28 * px + self.b * 16 * px          # y_hat 12 + y_comp 12 + v_map 4 (+ target 12, v_target 4 per sample)
        l1b = n * 52 * px + self.b * 16 * px          # + the two gradients written (24)
        return [("mt_warp_fwd", 1, n * 36 * px + self.b * 4 * px, "hbm"),
                ("mt_chn_pack", 1, n * 56 * px + self.b * 16 * px, "hbm"),
                ("mt_chn_composite_fwd", 1, n * 36 * px + self.b * 16 * px, "hbm"),
                ("mt_chn_l1x3_fwd", 1, l1f, "hbm"), ("mt_chn_l1x3_bwd", 1, l1b, "hbm"),
                ("mt_chn_composite_bwd", 1, n * 48 * px + self.b * 4 * px, "hbm")]

    def sub(self, b):
        return Cfg5(b, self.f, self.h, self.w)


WORKLOADS = {"align": Align, "cfg1": Cfg1, "cfg2": Cfg2, "cfg3": Cfg3, "cfg4": Cfg4, "cfg5": Cfg5}


# ---------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML during the timed region."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown",
               0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting"}

    def __init__(self, device_index, period=0.003):
        super().__init__(daemon=True)
        self.period, self.samples, self.reasons, self.ok = period, [], set(), False
        self._halt = threading.Event()
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            self.nv = pynvml
            try:
                uuid = str(torch.cuda.get_device_properties(device_index).uuid)
                if not uuid.startswith("GPU-"):
                    uuid = "GPU-" + uuid
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception as e:           # noqa: BLE001
            log("clock sampling unavailable:", e)
            self.max_mhz = None

    def sample(self):
        if not self.ok:
            return
        try:
            self.samples.append(int(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
            try:
                bits = int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                bits = int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            for bit, name in self.REASONS.items():
                if bits & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def run(self):
        while not self._halt.is_set():
            self.sample()
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        if self.is_alive():
            self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}



def bind_to_gpu_numa(device_index):
    """Pins this rank to the CPUs NVML reports as local to its GPU BEFORE any pinned host buffer is allocated, so
    that first-touch places the staging buffers on the GPU's NUMA node (N ranks on one node otherwise share
    whatever node the launcher started them on).  Returns a short description for the JSON line."""
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(device_index).uuid)
            h = pynvml.nvmlDeviceGetHandleByUUID(uuid if uuid.startswith("GPU-") else "GPU-" + uuid)
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        allowed = os.sched_getaffinity(0)
        cpus = sorted(cpus & allowed)
        if not cpus:
            return {"bound": False, "why": "NVML reports no local CPU inside this process's cpuset"}
        os.sched_setaffinity(0, cpus)
        node = None
        try:
            for n in sorted(os.listdir("/sys/devices/system/node")):
                if n.startswith("node") and n[4:].isdigit():
                    lst = open("/sys/devices/system/node/%s/cpulist" % n).read().strip()
                    ids = set()
                    for part in lst.split(","):
                        if part:
                            lo, _, hi = part.partition("-")
                            ids.update(range(int(lo), int(hi or lo) + 1))
                    if cpus[0] in ids:
                        node = int(n[4:])
        except Exception:
            pass
        return {"bound": True, "cpus": "%d-%d (%d)" % (cpus[0], cpus[-1], len(cpus)), "numa_node": node}
    except Exception as e:      # noqa: BLE001
        return {"bound": False, "why": str(e)[:80]}

# ---------------------------------------------------------------------------
# CPU arms
# ---------------------------------------------------------------------------
def cpu_time_workload(wl, seconds, threads=None, min_reps=2, max_reps=100000):
    """Times the torch-CPU port of the path (oracle/torch_port.py) on a bounded sample."""
    import torch
    from oracle import torch_port as tp
    if threads:
        torch.set_num_threads(threads)
    d = {k: torch.from_numpy(v) for k, v in wl.host_inputs(1234).items()}
    wl.cpu_step(tp, d)                       # warm-up
    times, t_end = [], time.perf_counter() + seconds
    while len(times) < min_reps or (time.perf_counter() < t_end and len(times) < max_reps):
        t0 = time.perf_counter()
        wl.cpu_step(tp, d)
        times.append(time.perf_counter() - t0)
    mean = sum(times) / len(times)
    return wl.frames_per_step / mean, mean, len(times), torch.get_num_threads()


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (torch-CPU port of
    its call sequence; the Python reference itself cannot travel to the GPU box)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    from oracle import torch_port as tp
    wl = WORKLOADS[args.workload]()
    # bounded sample: shrink the batch until (steps + warmup) steps fit in ~150 s
    d = {k: torch.from_numpy(v) for k, v in wl.host_inputs(1234).items()}
    t0 = time.perf_counter()
    wl.cpu_step(tp, d)
    t1 = time.perf_counter() - t0
    budget = 150.0
    b = wl.b
    while b > 1 and (args.steps + args.warmup) * t1 * (b / wl.b) > budget:
        b = max(1, b // 2)
    sample = wl.sub(b)
    d = {k: torch.from_numpy(v) for k, v in sample.host_inputs(1234).items()}
    for _ in range(args.warmup):
        sample.cpu_step(tp, d)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        sample.cpu_step(tp, d)
    dt = time.perf_counter() - t0
    value = sample.frames_per_step * args.steps / dt
    line = {
        "impl": "reference", "metric": "aligned_frames_per_sec", "value": value, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl.describe},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": torch.get_num_threads(),
                         "kind": "port",
                         "sample": "%s at batch_size=%d (%d aligned frames per step), torch %s CPU"
                                   % (wl.name, b, sample.frames_per_step, torch.__version__)},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    OUT.emit(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    affinity = bind_to_gpu_numa(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL_DEBUG is left as the caller set it: fd 1 is redirected to stderr for the whole run (_RealStdout),
        # so communicator banners cannot reach the JSON line
        dist.init_process_group("nccl", device_id=dev)

    import master_thesis_b200 as mtb
    from master_thesis_b200 import _lib, ops
    _lib.load()
    wl = WORKLOADS[args.workload](args.batch) if args.batch > 0 else WORKLOADS[args.workload]()
    hbm_peak, tf_peak, peak_src = measured_peaks()

    # The job is world x (per-GPU batch) samples; rank r owns the contiguous block shard.batch_shard gives it
    # (SURVEY 8e: samples / (b, f) frames are independent, no data-path collective).  The synthetic samples of a
    # block are generated from its first global sample index, so the job's data does not depend on how many
    # ranks run it.  Input sets rotate so that every step reads inputs last touched >= 2 steps ago.
    from master_thesis_b200 import shard
    s_lo, s_hi = shard.batch_shard(wl.b * world, rank, world)
    assert s_hi - s_lo == wl.b
    nsets = args.sets
    host_sets = [wl.host_inputs(1000 * (s_lo // wl.b) + 17 * i) for i in range(nsets)]
    dsets = [{k: torch.from_numpy(v).to(dev) for k, v in hs.items()} for hs in host_sets]
    plans, outs, graphs = [], [], []
    for d in dsets:
        with ops.record() as plan:
            outs.append(wl.gpu_step(mtb, d))
        plans.append(plan)
    torch.cuda.synchronize()
    calls = wl.calls(plans[0]) if wl.name == "cfg3" else wl.calls()
    step_bytes = sum(c[2] for c in calls)
    use_graph = args.graph and getattr(wl, "graph_ok", True)
    if use_graph:
        # the same step captured as a CUDA graph: one launch per step instead of one foreign
        # call per kernel (small configs are host-issue-bound otherwise)
        for d in dsets:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                outs.append(wl.gpu_step(mtb, d))
            graphs.append(g)
    names = plans[0].names()
    # group the recorded launches by C-ABI call
    assert names == [c[0] for c in calls], (names, calls)
    launches_per_step = sum(c[1] for c in calls)
    torch.cuda.synchronize()

    ddp = None
    if args.ddp_mb > 0 and world > 1:
        # the only collective of the reference: DDP's gradient all-reduce (NCCL over NVLink), issued next to the
        # hot-path kernels of the step on its own stream in 25 MB buckets, as DDP does (SURVEY section 5)
        nfloat = int(args.ddp_mb * 1e6 / 4)
        ddp = {"grads": torch.zeros(nfloat, device=dev), "stream": torch.cuda.Stream(device=dev),
               "bucket": int(25e6 / 4), "bytes": nfloat * 4}

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def one_step(i):
        if ddp:
            # DDP overlaps the all-reduce of the buckets that are ready with the rest of the backward pass: here
            # the collective of step i runs concurrently with the hot-path kernels of step i (they are independent)
            main = torch.cuda.current_stream(dev)
            ddp["stream"].wait_stream(main)
            with torch.cuda.stream(ddp["stream"]):
                g = ddp["grads"]
                for o in range(0, g.numel(), ddp["bucket"]):
                    dist.all_reduce(g[o:o + ddp["bucket"]])
        if graphs:
            graphs[i % nsets].replay()
        else:
            plans[i % nsets]()
        if ddp:
            torch.cuda.current_stream(dev).wait_stream(ddp["stream"])

    for i in range(max(args.warmup, 3)):
        plans[i % nsets]()
        one_step(i)
    barrier()

    K = args.steps

    def timed_round():
        """EXACTLY K steps between two events, barrier + synchronize on both sides, max over ranks."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            one_step(i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    # by default the timed region is run once; with --min-ms it is repeated until that much device time has been
    # integrated (a 20-step run of a 100 us step is 2 ms: too short for the clock sampler and at the mercy of one
    # stray interrupt); every repetition times exactly K steps, the reported one is the median
    sampler = ClockSampler(local)
    sampler.start()
    # one untimed pass over the same K steps first (counted in the line's "warmup"): after the --warmup steps, the
    # first back-to-back pass still ran ~25 us slower in all, with or without the clock sampler (align, 20 steps on
    # one B200 at 1000 W, two runs: 90.4 / 90.3 against medians of 89.0 / 89.1 us per step; after this pass the
    # first timed pass ran at 89.1 / 89.0)
    timed_round()
    first = timed_round()
    n_rounds = int(min(args.max_rounds, max(1, -(-args.min_ms // max(first, 1e-3)))))
    if world > 1:                 # every rank must run the same number of rounds (they contain barriers)
        t = torch.tensor([n_rounds], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        n_rounds = int(t.item())
    rounds = [first] + [timed_round() for _ in range(n_rounds - 1)]
    ms = sorted(rounds)[len(rounds) // 2]
    value = wl.frames_per_step * world * K / (ms * 1e-3)
    # the results of the last timed step (step K - 1 used input set (K - 1) % nsets), copied on the device before
    # anything else runs; written out at the end so that the host work stays outside every timed region
    last = None
    if args.dump_outputs and rank == 0:
        last, skipped = result_tensors(outs[nsets + (K - 1) % nsets] if graphs else outs[(K - 1) % nsets])
        last = {k: t.detach().clone() for k, t in last.items()}
        if skipped:
            log("--dump-outputs: not tensors, not written:", ", ".join(skipped))

    # one more repetition of the same K steps, instrumented: one event after every C-ABI call (individual
    # launches instead of the graph replay, so each interval also carries the launch gap that back-to-back
    # launches hide: the per-kernel figures below are conservative)
    ev = []
    barrier()
    ei0, ei1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ei0.record()
    for i in range(K):
        plan = plans[i % nsets]
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(calls) + 1)]
        evs[0].record()
        for j in range(len(calls)):
            plan.run_entry(j)
            evs[j + 1].record()
        ev.append(evs)
    ei1.record()
    sampler.sample()
    barrier()
    clocks = sampler.stop()
    ms_instr = ei0.elapsed_time(ei1)

    # per-call device time inside that timed region
    per_call = []
    cnames = [c[0] for c in calls]
    for j, c in enumerate(calls):
        cname, nl, nbytes, bound = c[:4]
        ts = [evs[j].elapsed_time(evs[j + 1]) for evs in ev]
        avg = sum(ts) / len(ts)
        ent = {"call": cname if cnames.count(cname) == 1 else "%s#%d" % (cname, j),
               "launches": nl, "avg_us": 1e3 * avg, "bound": bound,
               "algorithmic_bytes": nbytes, "achieved_gbs": nbytes / (avg * 1e-3) / 1e9,
               "frac_hbm": nbytes / (avg * 1e-3) / 1e9 / hbm_peak}
        if bound == "tensor":
            ent["flop"] = c[4]
            ent["achieved_tflops"] = c[4] / (avg * 1e-3) / 1e12
        per_call.append(ent)
    traffic_all = {}
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(traffic_file) and args.batch <= 0:
        try:
            traffic_all = json.load(open(traffic_file)).get(args.workload, {})
        except Exception:
            traffic_all = {}
    for ent in per_call:
        t = traffic_all.get(ent["call"]) or traffic_all.get(ent["call"].split("#")[0])
        if t:
            ent["kernel"], ent["traffic"] = t.get("kernel"), t.get("traffic")
    # dominant kernel = largest device time per LAUNCH among the HBM-bound calls; prefer single-launch calls,
    # whose event interval is exactly one kernel (multi-launch calls are listed under "kernels")
    hbm_calls = [c for c in per_call if c["bound"] == "hbm"]
    single = [c for c in hbm_calls if c["launches"] == 1] or hbm_calls or per_call
    dom = max(single, key=lambda c: c["avg_us"] / c["launches"])
    call = dom["call"].split("#")[0]
    kname = {"mt_warp_fwd": "warp_fwd_kernel", "mt_warp_pack_fwd": "warp_fwd_kernel<PACK>",
             "mt_warp_l1_fwd": "warp_l1_fwd_kernel", "mt_warp_l1_bwd": "warp_l1_bwd_kernel"}.get(call, call)
    roofline = {"bound": "hbm", "kernel": dom.get("kernel") or kname, "call": dom["call"],
                "launches_in_call": dom["launches"],
                "achieved": dom["achieved_gbs"], "peak": hbm_peak, "unit": "GB/s",
                "frac": dom["frac_hbm"], "traffic": dom.get("traffic"), "peak_source": peak_src,
                "avg_us": dom["avg_us"], "algorithmic_bytes": dom["algorithmic_bytes"],
                "timing": "CUDA events around every C-ABI call of the instrumented repetition of the timed region"}
    line_extra = {}
    tc = [c for c in per_call if c["bound"] == "tensor"]
    if tc:
        # the tcgen05 correlation: a dense contraction that is bandwidth-bound from cold HBM (AI 73 flop/B at F=4,
        # ridge 252): achieved TFLOP/s against the measured bf16 peak, its HBM fraction, and the ncu pipe-active
        # counter of the committed capture of this kernel
        t0 = max(tc, key=lambda c: c["avg_us"])
        pipe = (traffic_all.get(t0["call"]) or traffic_all.get(t0["call"].split("#")[0]) or {})
        line_extra["roofline_tc"] = {
            "bound": "tensor", "kernel": pipe.get("kernel") or "corr_tc_kernel (tcgen05.mma kind::tf32, TMA, TMEM)",
            "call": t0["call"], "achieved": t0["achieved_tflops"], "peak": tf_peak, "unit": "TFLOP/s",
            "frac": t0["achieved_tflops"] / tf_peak, "peak_note": "measured dense bf16 cuBLAS peak; the kernel runs "
            "kind::tf32 (fp32 features consumed as they are), whose tensor-pipe rate is half of bf16",
            "hbm_frac": t0["frac_hbm"], "achieved_gbs": t0["achieved_gbs"], "avg_us": t0["avg_us"],
            "flop": t0["flop"], "algorithmic_bytes": t0["algorithmic_bytes"], "traffic": pipe.get("traffic"),
            "tensor_pipe_active_pct": pipe.get("tensor_pipe_active_pct"), "tensor_pipe_source": pipe.get("source")}

    # ---- end-to-end: pinned host inputs -> H2D -> kernels -> D2H, every step ----
    e2e = run_e2e(args, wl, mtb, ops, host_sets[0], dev, world)

    line = {
        "metric": "aligned_frames_per_sec", "value": value, "unit": "frames/s", "n_gpus": world,
        "steps": K, "warmup": max(args.warmup, 3) + K, "ms_per_step": ms / K, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl.describe, "frames_per_step_per_gpu": wl.frames_per_step,
                   "l2": "inputs rotate over %d buffer sets; %.0f MB algorithmic traffic per step, "
                         ">= %.0f MB between reuses of a set (L2 = 126 MB)"
                         % (nsets, step_bytes / 1e6, (nsets - 1) * step_bytes / 1e6),
                   "sharding": "shard.batch_shard: contiguous blocks of %d of the job's %d samples per rank, %d ranks, "
                               "no data-path collective" % (wl.b, wl.b * world, world),
                   "launch": "CUDA graph replay per step" if graphs else "one C-ABI call per kernel group",
                   "timed_region": "%d repetitions of exactly %d steps (barrier + sync around each) after %d warm-up "
                                   "steps and one untimed pass of the %d steps (\"warmup\" counts both); value = the "
                                   "median repetition" % (len(rounds), K, max(args.warmup, 3), K)},
        "rounds_ms": {"n": len(rounds), "min": min(rounds), "median": ms, "max": max(rounds),
                      "integrated_ms": sum(rounds), "instrumented": ms_instr},
        "clocks": clocks, "e2e": e2e, "host_affinity": affinity, "gpu_launches": launches_per_step * K,
        "roofline": roofline, "kernels": per_call,
    }
    line.update(line_extra)
    if ddp:
        # the collective alone and the kernels alone, for reading the overlap: step ~ max(kernels, all-reduce) when they overlap
        def ar_only():
            g = ddp["grads"]
            for o in range(0, g.numel(), ddp["bucket"]):
                dist.all_reduce(g[o:o + ddp["bucket"]])
        for _ in range(3):
            ar_only()
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(10):
            ar_only()
        a1.record()
        barrier()
        ar_ms = a0.elapsed_time(a1) / 10
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        for i in range(K):
            (graphs[i % nsets].replay() if graphs else plans[i % nsets]())
        k1.record()
        barrier()
        kern_ms = k0.elapsed_time(k1) / K
        t = torch.tensor([ar_ms, kern_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ar_ms, kern_ms = float(t[0]), float(t[1])
        line["ddp"] = {"allreduce_bytes_per_step": ddp["bytes"], "bucket_bytes": ddp["bucket"] * 4,
                       "allreduce_alone_ms": ar_ms, "kernels_alone_ms_per_step": kern_ms,
                       "value_without_allreduce": wl.frames_per_step * world / (kern_ms * 1e-3),
                       "allreduce_busbw_gbs": 2.0 * (world - 1) / world * ddp["bytes"] / (ar_ms * 1e-3) / 1e9,
                       "note": "NCCL all-reduce of a gradient-sized fp32 buffer (DFPN 13.92 M / CHN 14.69 M parameters, "
                               "SURVEY section 5) on its own stream inside every timed step, overlapped with the kernels"}
    if rank == 0 and world == 1 and hasattr(wl, "loop_stats"):
        line["loop"] = wl.loop_stats(mtb, dev)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sample = wl   # the full workload, repeated for about --cpu-seconds of CPU work
        v, mean, reps, cores = cpu_time_workload(sample, args.cpu_seconds)
        line["cpu_baseline"] = {
            "value": v, "unit": "frames/s", "cores": cores, "kind": "port",
            "sample": "%s at batch_size=%d: %d reps of %.3f s (torch %s CPU port of the reference "
                      "call sequence)" % (wl.name, sample.b, reps, mean, torch.__version__)}
    if last is not None:
        line["dumped_outputs"] = dump_outputs(last, args.dump_outputs)
    if rank == 0:
        OUT.emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


DUMP_BYTES = 60_000_000      # all .npy files of --dump-outputs together (the limit is 64 MB; headroom for headers)


def result_tensors(step_out):
    """The tensors of a step's result dict by name: a tuple or list entry (cfg5's "keep", the intermediates its step
    also returns) becomes <name>_<i>.  Returns (tensors, names of the entries that are not tensors)."""
    import torch
    tensors, skipped = {}, []
    for k, v in step_out.items():
        for name, t in ([("%s_%d" % (k, i), e) for i, e in enumerate(v)] if isinstance(v, (tuple, list))
                        else [(k, v)]):
            if isinstance(t, torch.Tensor):
                tensors[name] = t
            else:
                skipped.append(name)
    return tensors, skipped


def dump_outputs(tensors, directory):
    """Writes every tensor as <directory>/<name>.npy: float64 for 64-bit floats and for integers (exact), float32
    otherwise.  The byte budget is shared out from the smallest array up; an array larger than its share is
    replaced by a fixed sample of its elements: the flattened array at the sorted indices that
    numpy.random.default_rng(0) draws without replacement, so two runs on the same shapes sample the same
    elements.  Returns {name: [shape, number of elements written]}."""
    import numpy as np
    import torch
    os.makedirs(directory, exist_ok=True)
    written, left = {}, DUMP_BYTES
    items = sorted(tensors.items(), key=lambda kv: (kv[1].numel(), kv[0]))
    for i, (name, t) in enumerate(items):
        wide = t.dtype == torch.float64 or not (t.is_floating_point() or t.dtype == torch.bool)
        dtype = torch.float64 if wide else torch.float32
        share = left // (len(items) - i) // (8 if wide else 4)
        if t.numel() > share:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), share, replace=False))
            t_out = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        else:
            t_out = t
        a = t_out.to(dtype).cpu().numpy()
        np.save(os.path.join(directory, name + ".npy"), a)
        left -= a.nbytes
        written[name] = [list(t.shape), int(a.size)]
    return written


def run_e2e(args, wl, mtb, ops, host, dev, world):
    """Same metric through the public API with HOST buffers: every step copies its inputs
    from pinned host memory, runs the kernels, and copies every result back.  Two
    pipeline slots (streams) overlap step i+1's H2D with step i's D2H."""
    import torch
    import torch.distributed as dist
    slots = []
    for _ in range(2):
        st = torch.cuda.Stream(device=dev)
        pin_in = {k: torch.from_numpy(v).pin_memory() for k, v in host.items()}
        with torch.cuda.stream(st):
            d_in = {k: torch.empty_like(v, device=dev) for k, v in pin_in.items()}
            for k in d_in:
                d_in[k].copy_(pin_in[k], non_blocking=True)
            with ops.record() as plan:
                out = wl.gpu_step(mtb, d_in)
            out = {k: v for k, v in out.items() if isinstance(v, torch.Tensor)}   # results copied back
            pin_out = {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in out.items()}
        st.synchronize()
        slots.append((st, pin_in, d_in, plan, out, pin_out))
    h2d = sum(v.numel() * v.element_size() for v in slots[0][1].values())
    d2h = sum(v.numel() * v.element_size() for v in slots[0][5].values())
    K = min(args.steps, args.e2e_steps)

    def one(i):
        st, pin_in, d_in, plan, out, pin_out = slots[i % 2]
        with torch.cuda.stream(st):
            for k in pin_in:
                d_in[k].copy_(pin_in[k], non_blocking=True)
            plan()
            for k in out:
                pin_out[k].copy_(out[k], non_blocking=True)

    for i in range(4):
        one(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    main = torch.cuda.current_stream(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(main)
    for st, *_ in slots:
        st.wait_stream(main)
    for i in range(K):
        one(i)
    for st, *_ in slots:
        main.wait_stream(st)
    e1.record(main)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    # the platform's ceiling for this step: the same pinned copies on the same two streams, no kernels
    # (all ranks at once: at N > 1 they share the host's memory bandwidth and PCIe root ports)
    def copies_only(i):
        st, pin_in, d_in, plan, out, pin_out = slots[i % 2]
        with torch.cuda.stream(st):
            for k in pin_in:
                d_in[k].copy_(pin_in[k], non_blocking=True)
            for k in out:
                pin_out[k].copy_(out[k], non_blocking=True)

    Kc = max(2, min(K, 20))
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record(main)
    for st, *_ in slots:
        st.wait_stream(main)
    for i in range(Kc):
        copies_only(i)
    for st, *_ in slots:
        main.wait_stream(st)
    c1.record(main)
    torch.cuda.synchronize()
    ms_copy = c0.elapsed_time(c1)
    if world > 1:
        t = torch.tensor([ms_copy], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_copy = float(t.item())
    return {"value": wl.frames_per_step * world * K / (ms * 1e-3), "unit": "frames/s",
            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": K,
            "ms_per_step": ms / K,
            "copies_only_ms_per_step": ms_copy / Kc,
            "copies_only_gbs_per_rank": (h2d + d2h) / (ms_copy / Kc * 1e-3) / 1e9,
            "fraction_of_copy_ceiling": (ms_copy / Kc) / (ms / K),
            "api": "master_thesis_b200 plug-point mirrors on pinned host tensors, 2 pipelined streams"}


class _RealStdout(object):
    """Keeps stdout clean: fd 1 is pointed at stderr for the whole run (NCCL / libraries print
    banners on it) and the single JSON line is written to the saved, real stdout."""

    def __init__(self):
        sys.stdout.flush()
        self.fd = os.dup(1)
        os.dup2(2, 1)

    def emit(self, line):
        sys.stdout.flush()
        os.write(self.fd, (line + "\n").encode())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="align", choices=sorted(WORKLOADS))
    ap.add_argument("--min-ms", type=float, default=0.0,
                    help="repeat the timed region of exactly --steps steps until this much device time is integrated "
                         "and report the median repetition (default: one timed region)")
    ap.add_argument("--max-rounds", type=int, default=400)
    ap.add_argument("--ddp-mb", type=float, default=-1.0,
                    help="N > 1: all-reduce a gradient-sized fp32 buffer of this many MB next to every step (NCCL); "
                         "default: 55.7 for cfg3 (DFPN), 58.8 for cfg5 (CHN), none otherwise")
    ap.add_argument("--batch", type=int, default=0,
                    help="per-GPU batch size override (scaling experiments; 0 = the config's own)")
    ap.add_argument("--sets", type=int, default=3)
    ap.add_argument("--e2e-steps", type=int, default=100)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", dest="graph", action="store_false",
                    help="issue every step as individual C-ABI calls instead of a CUDA graph replay")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step as DIR/<name>.npy (rank 0; at most 64 MB in all, "
                         "larger results as a fixed seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's results; --impl reference runs a smaller batch on the CPU")
    if args.gpus > 1 and "RANK" not in os.environ and args.impl != "reference":
        # convenience: re-launch under torchrun (the driver launches torchrun itself)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
               "--nproc-per-node", str(args.gpus), "--master-addr", "127.0.0.1",
               "--master-port", str(29400 + os.getpid() % 500), os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    if args.ddp_mb < 0:
        args.ddp_mb = {"cfg3": 55.7, "cfg5": 58.8}.get(args.workload, 0.0)
    global OUT
    OUT = _RealStdout()
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
