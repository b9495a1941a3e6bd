#!/bin/bash
# warp kernels reduced to their shipped launch shapes: build, the whole GPU suite, smoke, then a same-call A/B of every
# bench workload against a build of the parent commit (same C ABI, selected with MT_B200_LIB), alternating the two
# libraries three times, and a bit-for-bit comparison of the outputs both dump
#   bash tools/gpu/run_ar.sh PARENT_LIB [output directory, default a new temporary directory]
cd "$(dirname "$0")/../.."
PARENT="$(realpath "$1")"
OUT="${2:-$(mktemp -d)}"
DUMP="$(mktemp -d)"
echo "outputs: $OUT"
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/ar_gpu.txt"
python -c "import __graft_entry__ as g; g.build()" || exit 1
timeout 900 python -m pytest tests -q -m gpu 2>&1 | tail -6 | tee "$OUT/ar_gputest.txt"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
bench() {  # library workload repeat [extra arguments]
    local lib=$1 wl=$2 rep=$3; shift 3
    if [ "$lib" = parent ]; then export MT_B200_LIB="$PARENT"; else unset MT_B200_LIB; fi
    timeout 600 python bench.py --workload "$wl" --no-cpu-baseline --e2e-steps 2 "$@" \
        > "$OUT/ar_${wl}_${lib}_$rep.json" 2> "$OUT/ar_${wl}_${lib}_$rep.err"
    echo "$wl $lib $rep rc=$?"
    unset MT_B200_LIB
}
for wl in align cfg1 cfg2 cfg3 cfg4 cfg5; do
    # the first repeat also dumps the last step's outputs (written after the timed and instrumented passes)
    bench parent "$wl" 1 --dump-outputs "$DUMP/parent_$wl"
    bench new "$wl" 1 --dump-outputs "$DUMP/new_$wl"
    bench new "$wl" 2
    bench parent "$wl" 2
    bench parent "$wl" 3
    bench new "$wl" 3
done
python - "$OUT" "$DUMP" <<'EOF' | tee "$OUT/ar_summary.txt"
import glob, json, os, statistics, sys
import numpy as np
out, dump = sys.argv[1:3]
summary = {}
for wl in ("align", "cfg1", "cfg2", "cfg3", "cfg4", "cfg5"):
    s = summary[wl] = {}
    for lib in ("parent", "new"):
        runs = []
        for rep in (1, 2, 3):
            try:
                runs.append(json.loads(open(os.path.join(out, "ar_%s_%s_%d.json" % (wl, lib, rep))).read().splitlines()[-1]))
            except Exception as e:
                print(wl, lib, rep, "no result:", e)
        ms = [1e3 * r["ms_per_step"] for r in runs]
        calls = {}
        for r in runs:
            for c in r["kernels"]:
                if "warp" in c["call"] or "corr" in c["call"]:
                    calls.setdefault(c["call"], []).append(c["avg_us"])
        s[lib] = {"us_per_step": ms, "median": statistics.median(ms) if ms else None,
                  "spread": max(ms) - min(ms) if ms else None,
                  "calls_median_us": {k: statistics.median(v) for k, v in calls.items()}}
    pd, nd = os.path.join(dump, "parent_" + wl), os.path.join(dump, "new_" + wl)
    names = sorted(os.path.basename(p) for p in glob.glob(os.path.join(pd, "*.npy")))
    same = {}
    for n in names:
        a, b = np.load(os.path.join(pd, n)), np.load(os.path.join(nd, n)) if os.path.exists(os.path.join(nd, n)) else None
        same[n] = b is not None and a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()
    s["dump"] = {"arrays": len(names), "identical": sum(same.values()),
                 "different": [n for n, v in same.items() if not v],
                 "only_new": sorted(set(os.listdir(nd)) - set(names)) if os.path.isdir(nd) else None}
    p, n = s["parent"], s["new"]
    print("%-5s step us parent %s new %s | median %.2f / %.2f, spread %.2f / %.2f | dump %d/%d identical %s" % (
        wl, ["%.2f" % v for v in p["us_per_step"]], ["%.2f" % v for v in n["us_per_step"]], p["median"] or 0,
        n["median"] or 0, p["spread"] or 0, n["spread"] or 0, s["dump"]["identical"], s["dump"]["arrays"],
        s["dump"]["different"] or ""))
    for k in sorted(set(p["calls_median_us"]) | set(n["calls_median_us"])):
        print("      %-28s %8.2f %8.2f" % (k, p["calls_median_us"].get(k, float("nan")), n["calls_median_us"].get(k, float("nan"))))
json.dump(summary, open(os.path.join(out, "ar_summary.json"), "w"), indent=1)
EOF
rm -rf "$DUMP"
