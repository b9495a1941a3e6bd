#!/bin/bash
# batched clip inpainting: build, batched-inpainting tests, the whole GPU suite, smoke, bench lines, loop- and kernel-level timing
#   bash tools/gpu/run_ap.sh [output directory, default a new temporary directory]
cd "$(dirname "$0")/../.."
OUT="${1:-$(mktemp -d)}"
echo "outputs: $OUT"
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" || exit 1
timeout 900 python -m pytest tests/test_inpaint_batched.py -q -m gpu 2>&1 | tail -25 | tee "$OUT/ap_batched_tests.txt"
timeout 1200 python -m pytest tests -q -m gpu 2>&1 | tail -4 | tee "$OUT/ap_gputest.txt"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
timeout 300 python bench.py --gpus 1 --steps 50 --warmup 5 > "$OUT/ap_bench_align.json" 2>/dev/null; tail -c 400 "$OUT/ap_bench_align.json"
timeout 600 python bench.py --gpus 1 --steps 50 --warmup 5 --workload cfg4 > "$OUT/ap_bench_cfg4.json" 2>/dev/null; tail -c 600 "$OUT/ap_bench_cfg4.json"
timeout 900 python tools/gpu/time_inpaint_batched.py "$OUT/ap_time_inpaint.json" 2>&1 | grep '^{"'
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/ap_gpu.txt"
