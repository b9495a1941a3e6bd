#!/bin/bash
# resize kernels (F5): build, resize tests, the whole GPU suite, smoke, bench line, eager-vs-kernel timing at cfg3
#   bash tools/gpu/run_ao.sh [output directory, default a new temporary directory]
cd "$(dirname "$0")/../.."
OUT="${1:-$(mktemp -d)}"
echo "outputs: $OUT"
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" || exit 1
timeout 600 python -m pytest tests/test_resize.py -q -m gpu 2>&1 | tail -25 | tee "$OUT/ao_resize_tests.txt"
timeout 900 python -m pytest tests -q -m gpu 2>&1 | tail -4 | tee "$OUT/ao_gputest.txt"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
timeout 300 python bench.py --gpus 1 --steps 50 --warmup 5 > "$OUT/ao_bench_align.json" 2>/dev/null; tail -c 400 "$OUT/ao_bench_align.json"
timeout 600 python tools/gpu/time_resize.py "$OUT/ao_time_resize.json" 2>&1 | grep '^{"call"'
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/ao_gpu.txt"
