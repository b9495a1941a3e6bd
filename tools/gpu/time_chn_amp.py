"""Mixed-precision CHN: the composite and fill kernels reading a half RRDBNet output natively, against the fp32
kernels, and against what a user would otherwise write under autocast (an eager ``.float()`` of the half output, the
fp32 kernel, and for the backward the cast of the fp32 gradient back to half).

Arms, per workload:
  fp32    fp32 nn_out, the fp32 entry points
  <dt>    fp16 / bf16 nn_out read by the *_dt entry points (gradient written in the half dtype)
  <dt>+cast  the same half nn_out copied to fp32 by an eager cast, the fp32 entry points, the fp32 gradient cast back
Workloads: composite forward + backward (g_yhat and g_comp) at B = 8 and 32, F = 4, 256 x 256 (cfg5 sizes);
mt_chn_fill_step at B = 1, 480 x 854; mt_chn_fill_lanes at L = 8, 480 x 854.

Every arm is one CUDA graph of REPS passes over K input sets whose total size exceeds twice the 126 MB L2, so each
pass reads its operands from HBM.  CUDA events around graph replays; the arms alternate, ROUNDS times, and the median
per arm is reported.  The fp32 arm's nn_out is the half nn_out widened, so every arm computes the same numbers: the
outputs of all arms are compared bit for bit in the same run (the fp32 arm's gradient after rounding to the half
dtype).  ``model_bytes_per_px`` is the algorithmic traffic per pixel and frame (computed, not measured), with x_t and v_t
of the composite counted for every frame although the F frames of a sample re-read them from L2: ``model_GBps`` is
therefore an upper bound of the HBM rate, not a measured one.

    python tools/gpu/time_chn_amp.py [out.json]
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


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                                       "-i", str(torch.cuda.current_device())], text=True, timeout=30).strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except (OSError, subprocess.SubprocessError, ValueError):
        return {"name": torch.cuda.get_device_name(), "power_limit": "unknown", "max_sm_clock": "unknown"}


def p(t):
    return ops._ptr(t)


def n_sets(bytes_per_set):
    return max(2, -(-2 * L2_BYTES // bytes_per_set) + 1)


def composite_sets(b, f, h, w, dt):
    """Input / output buffers of one composite forward + backward: nn_out in the half dtype and widened."""
    P = h * w
    g = torch.Generator(device="cuda").manual_seed(b * 7 + f)

    def rnd(*shape):
        return torch.randn(shape, generator=g, device="cuda")
    sets = []
    per_set = b * f * 3 * P * (4 + 2 + 4 * 2 + 4 * 2 + 4 + 2 + 4 + 2)
    for _ in range(n_sets(per_set)):
        nn_h = rnd(b * f, 3, h, w).to(dt)
        s = dict(nn_h=nn_h, nn32=nn_h.float(), nn32c=torch.empty(b * f, 3, h, w, device="cuda"),
                 x_t=torch.rand(b, 3, h, w, generator=g, device="cuda"),
                 v_t=(torch.rand(b, 1, h, w, generator=g, device="cuda") < 0.6).float(),
                 gy=rnd(b, 3, f, h, w), gc=rnd(b, 3, f, h, w))
        for arm in ("fp32", "half", "cast"):
            s["yh_" + arm] = torch.empty(b, f, 3, h, w, device="cuda")
            s["yc_" + arm] = torch.empty(b, f, 3, h, w, device="cuda")
        s["g_fp32"] = torch.empty(b * f, 3, h, w, device="cuda")
        s["g_half"] = torch.empty(b * f, 3, h, w, device="cuda", dtype=dt)
        s["g32_cast"] = torch.empty(b * f, 3, h, w, device="cuda")
        s["g_cast"] = torch.empty(b * f, 3, h, w, device="cuda", dtype=dt)
        sets.append(s)
    return sets


def composite_step(arm, s, b, f, P, code, st):
    nn, c = {"fp32": (s["nn32"], 0), "half": (s["nn_h"], code), "cast": (s["nn32c"], 0)}[arm]
    if arm == "cast":
        s["nn32c"].copy_(s["nn_h"])                                    # nn_out.float()
    _lib.call("mt_chn_composite_fwd_dt", c, p(nn), p(s["x_t"]), 3 * P, P, p(s["v_t"]), P, p(s["yh_" + arm]),
              p(s["yc_" + arm]), b, f, P, st)
    gs = s["gy"].stride()[:3]
    g = s["g32_cast"] if arm == "cast" else s["g_" + arm]
    _lib.call("mt_chn_composite_bwd_dt", c, p(nn), p(s["v_t"]), P, p(s["gy"]), *gs, p(s["gc"]), *gs, p(g), b, f, P, st)
    if arm == "cast":
        s["g_cast"].copy_(s["g32_cast"])                               # autograd's cast of the gradient back to half


def composite_check(sets):
    for s in sets:
        for arm in ("half", "cast"):
            assert torch.equal(s["yh_" + arm], s["yh_fp32"]) and torch.equal(s["yc_" + arm], s["yc_fp32"]), arm
        assert torch.equal(s["g_half"], s["g_cast"]) and torch.equal(s["g_half"], s["g_fp32"].to(s["g_half"].dtype))


def fill_sets(L, h, w, dt, lanes):
    P = h * w
    g = torch.Generator(device="cuda").manual_seed(L * 11 + int(lanes))
    sets = []
    per_set = L * P * (12 + 6 + 12 + 12 + 4 * 4 + 3 * (12 + 4 + 12))
    for _ in range(n_sets(per_set)):
        nn_h = torch.randn(L, 3, h, w, generator=g, device="cuda").to(dt)
        m_t = (torch.rand(L, 1, h, w, generator=g, device="cuda") < 0.3).float()
        s = dict(nn_h=nn_h, nn32=nn_h.float(), nn32c=torch.empty(L, 3, h, w, device="cuda"), m_t=m_t, v_t=1 - m_t,
                 x_t=torch.rand(L, 3, h, w, generator=g, device="cuda"),
                 v_map0=m_t * (torch.rand(L, 1, h, w, generator=g, device="cuda") < 0.5).float())
        for arm in ("fp32", "half", "cast"):
            s["out_" + arm] = [torch.empty(L, 3, h, w, device="cuda"), torch.empty(L, 1, h, w, device="cuda"),
                               torch.empty(L, 3, h, w, device="cuda"), torch.empty(L, device="cuda")]
        sets.append(s)
    return sets


def fill_step(arm, s, L, P, code, st, ws, slots):
    nn, c = {"fp32": (s["nn32"], 0), "half": (s["nn_h"], code), "cast": (s["nn32c"], 0)}[arm]
    if arm == "cast":
        s["nn32c"].copy_(s["nn_h"])
    y, m, x, per = s["out_" + arm]
    if slots is None:           # mt_chn_fill_step at B = L (= 1 here)
        _lib.call("mt_chn_fill_step_dt", c, p(nn), p(s["x_t"]), 3 * P, P, p(s["v_t"]), P, p(s["m_t"]), P,
                  p(s["v_map0"]), P, p(y), p(m), p(x), p(per), p(ws), L, P, st)
    else:
        _lib.call("mt_chn_fill_lanes_dt", c, p(nn), p(s["x_t"]), 3 * P, P, p(s["m_t"]), P, p(s["v_map0"]), P,
                  p(slots), p(y), 3 * P, P, p(m), P, p(x), 3 * P, P, p(per), p(ws), L, P, 0, 1.0, 0, st)


def fill_check(sets):
    for s in sets:
        for arm in ("half", "cast"):
            for a, b in zip(s["out_" + arm], s["out_fp32"]):
                assert a.data_ptr() != b.data_ptr() and torch.equal(a, b), arm


def time_arms(step, sets, arms):
    """{arm: median µs per pass} from CUDA graphs of REPS passes over all sets, arms alternating."""
    side = torch.cuda.Stream()
    graphs = {}
    with torch.cuda.stream(side):
        st = ops._stream(sets[0]["nn_h"])
        for arm in arms:                                   # eager warm-up: module load, first launches
            for s in sets:
                step(arm, s, st)
        side.synchronize()
        for arm in arms:
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr, stream=side):
                st = ops._stream(sets[0]["nn_h"])
                for _ in range(REPS):
                    for s in sets:
                        step(arm, s, st)
            graphs[arm] = gr
    torch.cuda.synchronize()
    times = {arm: [] for arm in arms}
    for arm in arms:
        graphs[arm].replay()
    torch.cuda.synchronize()
    for _ in range(ROUNDS):
        for arm in arms:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            graphs[arm].replay()
            e1.record()
            torch.cuda.synchronize()
            times[arm].append(e0.elapsed_time(e1) * 1e3 / (REPS * len(sets)))
    return {arm: statistics.median(v) for arm, v in times.items()}, {arm: v for arm, v in times.items()}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    assert torch.cuda.is_available(), "needs the GPU"
    _lib.load()
    result = {"card": card(), "l2_rotation": "K input sets per pass, K * set bytes > 2 x 126 MB",
              "reps_per_graph": REPS, "rounds": ROUNDS, "unit": "us per pass (median over rounds)", "workloads": []}
    ws = torch.zeros(int(_lib.load().mt_workspace_bytes()), dtype=torch.uint8, device="cuda")
    lws = torch.zeros(int(_lib.load().mt_chn_fill_lanes_workspace_bytes(8)), dtype=torch.uint8, device="cuda")
    for name, dt in HALVES.items():
        code = ops._DT[dt]
        for b in (8, 32):
            f, h, w = 4, 256, 256
            sets = composite_sets(b, f, h, w, dt)
            med, raw = time_arms(lambda arm, s, st: composite_step(arm, s, b, f, h * w, code, st), sets,
                                 ("fp32", "half", "cast"))
            composite_check(sets)
            px = b * f * h * w
            model = {"fp32": 104, "half": 86, "cast": 140}
            result["workloads"].append(dict(
                workload="composite fwd+bwd", dtype=name, B=b, F=f, H=h, W=w, sets=len(sets), us=med, rounds_us=raw,
                model_bytes_per_px=model, model_GBps={a: model[a] * px / (med[a] * 1e-6) / 1e9 for a in med},
                outputs_equal=True))
            del sets
            torch.cuda.empty_cache()
        for L, lanes in ((1, False), (8, True)):
            h, w = 480, 854
            sets = fill_sets(L, h, w, dt, lanes)
            slots = torch.arange(L, dtype=torch.int32, device="cuda") if lanes else None
            wsp = lws if lanes else ws
            med, raw = time_arms(lambda arm, s, st: fill_step(arm, s, L, h * w, code, st, wsp, slots), sets,
                                 ("fp32", "half", "cast"))
            fill_check(sets)
            px = L * h * w
            model = {"fp32": 60, "half": 54, "cast": 78} if lanes else {"fp32": 64, "half": 58, "cast": 82}
            result["workloads"].append(dict(
                workload="chn_fill_lanes" if lanes else "chn_fill", dtype=name, L=L, H=h, W=w, sets=len(sets), us=med,
                rounds_us=raw, model_bytes_per_px=model,
                model_GBps={a: model[a] * px / (med[a] * 1e-6) / 1e9 for a in med}, outputs_equal=True))
            del sets
            torch.cuda.empty_cache()
    for r in result["workloads"]:
        print(json.dumps({k: r[k] for k in ("workload", "dtype", "us") if k in r}))
    text = json.dumps(result, indent=1)
    if out_path:
        with open(out_path, "w") as fh:
            fh.write(text + "\n")
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
