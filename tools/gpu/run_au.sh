#!/bin/bash
# channels-last networks: build, tests/test_channels_last.py and the whole GPU suite, smoke, a same-call A/B of the
# default, cfg4 and cfg5 bench workloads against the parent commit (alternated three times) with a bit-for-bit
# comparison of both trees' --dump-outputs, then time_channels_last.py.  PARENT_TREE is a checkout of the parent commit
# with its library built.
#   bash tools/gpu/run_au.sh PARENT_TREE [output directory, default a new temporary directory]
cd "$(dirname "$0")/../.."
PARENT="$(realpath "$1")"
OUT="$(realpath -m "${2:-$(mktemp -d)}")"
DUMP="$(mktemp -d)"
echo "outputs: $OUT"
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/au_gpu.txt"
python -c "import __graft_entry__ as g; g.build()" || exit 1
timeout 900 python -m pytest tests/test_channels_last.py -q -m gpu -rf 2>&1 | grep -v "^\.*$" | tail -40 | tee "$OUT/au_cl_tests.txt"
timeout 1800 python -m pytest tests -q -m gpu --ignore=tests/test_channels_last.py -rf 2>&1 | tail -12 | tee "$OUT/au_gputest.txt"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2 | tee "$OUT/au_smoke.txt"
bench() {  # library workload repeat [extra arguments]
    local lib=$1 wl=$2 rep=$3 dir=.; shift 3
    if [ "$lib" = parent ]; then dir="$PARENT"; fi
    (cd "$dir" && timeout 600 python bench.py --workload "$wl" --no-cpu-baseline --e2e-steps 2 "$@" \
        > "$OUT/au_${wl}_${lib}_$rep.json" 2> "$OUT/au_${wl}_${lib}_$rep.err")
    echo "$wl $lib $rep rc=$?"
}
for wl in align cfg4 cfg5; do
    bench parent "$wl" 1 --dump-outputs "$DUMP/parent_$wl"
    bench new "$wl" 1 --dump-outputs "$DUMP/new_$wl"
    bench new "$wl" 2
    bench parent "$wl" 2
    bench parent "$wl" 3
    bench new "$wl" 3
done
python - "$OUT" "$DUMP" <<'PY' | tee "$OUT/au_summary.txt"
import glob, json, os, statistics, sys
import numpy as np
out, dump = sys.argv[1:3]
summary = {}
for wl in ("align", "cfg4", "cfg5"):
    s = summary[wl] = {}
    for lib in ("parent", "new"):
        ms = []
        for rep in (1, 2, 3):
            try:
                ms.append(1e3 * json.loads(open(os.path.join(out, "au_%s_%s_%d.json" % (wl, lib, rep))).read()
                                           .splitlines()[-1])["ms_per_step"])
            except Exception as e:
                print(wl, lib, rep, "no result:", e)
        s[lib] = {"us_per_step": ms, "median": statistics.median(ms) if ms else None,
                  "spread": max(ms) - min(ms) if ms else None}
    pd, nd = os.path.join(dump, "parent_" + wl), os.path.join(dump, "new_" + wl)
    names = sorted(os.path.basename(p) for p in glob.glob(os.path.join(pd, "*.npy")))
    same = {}
    for n in names:
        q = os.path.join(nd, n)
        a, b = np.load(os.path.join(pd, n)), (np.load(q) if os.path.exists(q) else None)
        same[n] = b is not None and a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()
    s["dump"] = {"arrays": len(names), "identical": sum(same.values()), "different": [n for n, v in same.items() if not v]}
    p, n = s["parent"], s["new"]
    print("%-5s step us parent %s new %s | median %.2f / %.2f, spread %.2f / %.2f | dump %d/%d identical %s" % (
        wl, ["%.2f" % v for v in p["us_per_step"]], ["%.2f" % v for v in n["us_per_step"]], p["median"] or 0,
        n["median"] or 0, p["spread"] or 0, n["spread"] or 0, s["dump"]["identical"], s["dump"]["arrays"],
        s["dump"]["different"] or ""))
json.dump(summary, open(os.path.join(out, "au_summary.json"), "w"), indent=1)
PY
rm -rf "$DUMP"
timeout 1500 python tools/gpu/time_channels_last.py "$OUT/r8_time_channels_last.json" 2>&1 | tail -30 | tee "$OUT/au_time.txt"
