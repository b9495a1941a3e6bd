"""Channels-last networks at the library boundary: what the layout copies cost, and what is left without them.

Arms, per row and precision (fp32, and bf16 under autocast):
  nchw        the network in the default NCHW layout, planar packs and planar reads (today's path)
  cl_copies   the network converted to channels_last, the library as before this change: planar pack, which the first
              convolution copies to NHWC; the NHWC output copied to planar for the composite / fill kernel; its planar
              gradient copied back to NHWC by the convolution's backward
  cl_native   the same channels-last network, the pack written and the output read in NHWC (this change)
Rows:
  chn_cfg5        CHN forward + backward at cfg5 sizes (B = 8, F = 4, 256 x 256): pack, network, composite forward
                  and backward with fixed upstream gradients
  fill_L1 / L8    the inference fill step at 480 x 854: warp + pack, network, fill (L = 1) / fill of 8 lanes
  flowest_cfg3    the DFPN FlowEstimator at 256 x 256, cfg3 sizes (B = 32, F = 4: 128 frames), forward + backward
                  w.r.t. the network weights and flow_pre
Each row is timed twice: "kernels" = the library's launches at the boundary alone (plus, in cl_copies, the layout
copies the network would make), "step" = the whole step with the network stand-in.

The networks are STAND-INS, not the reference's RRDBNet or FlowEstimator: a conv stack Conv2d(Cin, 32, 3) - ReLU -
Conv2d(32, Cout, 3) (Cin = 9 / 10, Cout = 3 / 2).  The real networks are far deeper, so their steps are much longer
and the copies a smaller share of them: the effect on the real networks is not measured here.

Every arm is one CUDA graph of K input sets whose inputs together exceed twice the 126 MB L2 (each replay reads its
inputs from HBM); CUDA events around REPS replays; the arms alternate ROUNDS times and the median per arm is reported.
Outputs of cl_copies and cl_native are compared bit for bit in the same run.

    python tools/gpu/time_channels_last.py [out.json]
"""
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from master_thesis_b200 import _lib, ops    # noqa: E402

L2_BYTES = 126 * 2 ** 20
REPS = 3
ROUNDS = 5
ARMS = ("nchw", "cl_copies", "cl_native")
CL = torch.channels_last


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


def stand_in(cin, cout, arm):
    torch.manual_seed(cin)
    net = nn.Sequential(nn.Conv2d(cin, 32, 3, padding=1), nn.ReLU(), nn.Conv2d(32, cout, 3, padding=1)).cuda()
    return net if arm == "nchw" else net.to(memory_format=CL)


def graph_of(fn, sets):
    """A CUDA graph of fn(s) over every input set (warmed up on a side stream first, as graph capture requires)."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            for s in sets:
                fn(s)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for s in sets:
            fn(s)
    torch.cuda.synchronize()
    return g


def us_per_step(g, n):
    g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(REPS):
        g.replay()
    b.record()
    b.synchronize()
    return 1e3 * a.elapsed_time(b) / (REPS * n)


# ---------------------------------------------------------------- rows
def chn_row(dt):
    b, f, h, w = 8, 4, 256, 256
    gen = torch.Generator(device="cuda").manual_seed(1)
    per_set = 4 * h * w * (b * 4 + b * f * (3 + 1 + 1) + 2 * b * f * 3)
    sets = []
    for _ in range(n_sets(per_set)):
        x_t = torch.rand(b, 3, h, w, generator=gen, device="cuda")
        v_t = (torch.rand(b, 1, h, w, generator=gen, device="cuda") < 0.6).float()
        x_al = torch.rand(b, 3, f, h, w, generator=gen, device="cuda")
        v_al = (torch.rand(b, 1, f, h, w, generator=gen, device="cuda") < 0.8).float()
        sets.append(dict(x_t=x_t, v_t=v_t, x_al=x_al, v_al=v_al, v_map=v_al * (1 - v_t.unsqueeze(2)),
                         gy=torch.randn(b, 3, f, h, w, generator=gen, device="cuda"),
                         gc=torch.randn(b, 3, f, h, w, generator=gen, device="cuda"),
                         nn_out=torch.randn(b * f, 3, h, w, generator=gen, device="cuda").to(dt)))
        sets[-1]["nn_out_cl"] = sets[-1]["nn_out"].contiguous(memory_format=CL)

    def kernels(arm):
        def fn(s):
            pack = ops.chn_pack(s["x_t"], s["v_t"], s["x_al"], s["v_al"], s["v_map"], channels_last=arm == "cl_native")
            no = s["nn_out" if arm == "nchw" else "nn_out_cl"]
            if arm == "cl_copies":
                pack.contiguous(memory_format=CL)       # the first convolution's input conversion
                no = no.contiguous()                     # the copy the composite made of the output
            ops.ChnCompositeFn.forward(_Ctx(), no, s["x_t"], s["v_t"], b, f)
            g = ops.chn_composite_bwd_raw(no, s["v_t"], s["gy"], s["gc"], b, f)
            if arm == "cl_copies":
                g.contiguous(memory_format=CL)           # the conversion of the planar gradient in the conv backward
            s["out_" + arm] = g
        return fn

    def step(arm):
        net = stand_in(9, 3, arm)

        def fn(s):
            with torch.autocast("cuda", dtype=dt, enabled=dt != torch.float32):
                pack = ops.chn_pack(s["x_t"], s["v_t"], s["x_al"], s["v_al"], s["v_map"],
                                    channels_last=arm == "cl_native")
                nn_out = net(pack)
                if arm == "cl_copies":
                    nn_out = nn_out.contiguous()
                yh, yc = ops.chn_composite(nn_out, s["x_t"], s["v_t"], b, f)
            torch.autograd.backward([yh, yc], [s["gy"], s["gc"]])
            s["step_" + arm] = yc
        return fn
    return sets, kernels, step


class _Ctx(object):
    def save_for_backward(self, *a):
        pass


def fill_row(dt, L):
    h, w = 480, 854
    gen = torch.Generator(device="cuda").manual_seed(2 + L)
    per_set = 4 * h * w * L * (3 + 1 + 3 + 1 + 2 + 1)
    sets = []
    for _ in range(n_sets(per_set)):
        x_t = torch.rand(L, 3, h, w, generator=gen, device="cuda")
        m_t = (torch.rand(L, 1, h, w, generator=gen, device="cuda") < 0.3).float()
        x_ref = torch.rand(L, 3, 1, h, w, generator=gen, device="cuda")
        m_ref = (torch.rand(L, 1, 1, h, w, generator=gen, device="cuda") < 0.3).float()
        base = torch.stack(torch.meshgrid(torch.linspace(-1, 1, w, device="cuda"), torch.linspace(-1, 1, h, device="cuda"),
                                          indexing="xy"), -1)
        flow = (base + 0.02 * torch.randn(L, 1, h, w, 2, generator=gen, device="cuda")).contiguous()
        st = [torch.zeros(sh, device="cuda") for sh in ((L, 3, h, w), (L, 1, h, w), (L, 3, h, w), (L,))]
        sets.append(dict(x_t=x_t, m_t=m_t, x_ref=x_ref, m_ref=m_ref, flow=flow, st=st,
                         nn_out=torch.randn(L, 3, h, w, generator=gen, device="cuda").to(dt)))
        sets[-1]["nn_out_cl"] = sets[-1]["nn_out"].contiguous(memory_format=CL)
    flags = ops.ALIGN_CORNERS | ops.VIS_FROM_MASK

    def fill(s, nn_out, v_map):
        if L == 1:
            return ops.chn_fill(nn_out, s["x_t"], 1 - s["m_t"], s["m_t"], v_map[:, :, 0])[0]
        ops.chn_fill_lanes(nn_out, s["x_t"], s["m_t"], v_map[:, :, 0], list(range(L)), *s["st"])
        return s["st"][2]

    def kernels(arm):
        def fn(s):
            nn_in, v_map, _, _ = ops.warp_pack_fwd(s["x_ref"], s["m_ref"], s["flow"], s["m_t"], s["x_t"], 1 - s["m_t"],
                                                   flags, channels_last=arm == "cl_native")
            no = s["nn_out" if arm == "nchw" else "nn_out_cl"]
            if arm == "cl_copies":
                nn_in.contiguous(memory_format=CL)
                no = no.contiguous()
            s["out_" + arm] = fill(s, no, v_map)
        return fn

    def step(arm):
        net = stand_in(9, 3, arm)

        def fn(s):
            with torch.no_grad(), torch.autocast("cuda", dtype=dt, enabled=dt != torch.float32):
                nn_in, v_map, _, _ = ops.warp_pack_fwd(s["x_ref"], s["m_ref"], s["flow"], s["m_t"], s["x_t"],
                                                       1 - s["m_t"], flags, channels_last=arm == "cl_native")
                nn_out = net(nn_in)
                if arm == "cl_copies":
                    nn_out = nn_out.contiguous()
                s["step_" + arm] = fill(s, nn_out, v_map)
        return fn
    return sets, kernels, step


def flowest_row(dt):
    b, f, h, w = 32, 4, 256, 256
    gen = torch.Generator(device="cuda").manual_seed(3)
    per_set = 4 * h * w * (b * 4 + b * f * 6)
    sets = []
    for _ in range(n_sets(per_set)):
        sets.append(dict(x_t=torch.rand(b, 3, h, w, generator=gen, device="cuda"),
                         m_t=(torch.rand(b, 1, h, w, generator=gen, device="cuda") < 0.3).float(),
                         x_r=torch.rand(b, 3, f, h, w, generator=gen, device="cuda"),
                         m_r=(torch.rand(b, 1, f, h, w, generator=gen, device="cuda") < 0.3).float(),
                         flow=torch.randn(b, f, h, w, 2, generator=gen, device="cuda").requires_grad_(True),
                         g=torch.randn(b, f, h, w, 2, generator=gen, device="cuda")))

    def kernels(arm):
        def fn(s):
            with torch.no_grad():
                nn_in = ops.flow_pack(s["x_t"], s["m_t"], s["x_r"], s["m_r"], s["flow"], channels_last=arm == "cl_native")
                if arm == "cl_copies":
                    nn_in = nn_in.contiguous(memory_format=CL)
            s["out_" + arm] = nn_in
        return fn

    def step(arm):
        net = stand_in(10, 2, arm)

        def fn(s):
            with torch.autocast("cuda", dtype=dt, enabled=dt != torch.float32):
                nn_in = ops.flow_pack(s["x_t"], s["m_t"], s["x_r"], s["m_r"], s["flow"],
                                      channels_last=arm == "cl_native")
                out = net(nn_in).reshape(b, f, 2, h, w).permute(0, 1, 3, 4, 2)
            out.backward(s["g"].to(out.dtype))
            s["step_" + arm] = out
        return fn
    return sets, kernels, step


def time_row(name, make, res):
    for dtn, dt in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
        sets, kernels, step = make(dt)
        row = res.setdefault(name, {}).setdefault(dtn, {"sets": len(sets)})
        for part, mk in (("kernels", kernels), ("step", step)):
            try:
                graphs = {arm: graph_of(mk(arm), sets) for arm in ARMS}
                times = {arm: [] for arm in ARMS}
                for _ in range(ROUNDS):
                    for arm in ARMS:
                        times[arm].append(us_per_step(graphs[arm], len(sets)))
                row[part] = {arm: {"median_us": statistics.median(v), "us": v} for arm, v in times.items()}
                key = ("out_" if part == "kernels" else "step_")
                a, c = sets[0][key + "cl_copies"], sets[0][key + "cl_native"]
                row[part]["cl_outputs_identical"] = bool(torch.equal(a, c))
                del graphs
            except Exception as e:      # one failing row must not lose the others
                row[part] = {"error": "%s: %s" % (type(e).__name__, e)}
            print(name, dtn, part, json.dumps({k: (v["median_us"] if isinstance(v, dict) and "median_us" in v else v)
                                               for k, v in row[part].items()}), flush=True)
        del sets
        torch.cuda.empty_cache()


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r8_time_channels_last.json")
    if not torch.cuda.is_available():
        raise SystemExit("time_channels_last.py needs a CUDA device")
    _lib.load()
    torch.backends.cudnn.benchmark = True
    res = {"card": card(), "reps": REPS, "rounds": ROUNDS, "L2_bytes": L2_BYTES,
           "stand_ins": "Conv2d(Cin,32,3)-ReLU-Conv2d(32,Cout,3); not the reference's RRDBNet / FlowEstimator",
           "rows": {}}
    time_row("chn_cfg5", chn_row, res["rows"])
    time_row("fill_L1", lambda dt: fill_row(dt, 1), res["rows"])
    time_row("fill_L8", lambda dt: fill_row(dt, 8), res["rows"])
    time_row("flowest_cfg3", flowest_row, res["rows"])
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as fh:
        json.dump(res, fh, indent=1)
    print("wrote", out)


if __name__ == "__main__":
    main()
