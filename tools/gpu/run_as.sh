#!/bin/bash
# mixed-precision DFPN aligner: build, the autocast tests, the whole GPU suite, smoke, the default bench line,
# time_dfpn_amp.py
#   bash tools/gpu/run_as.sh [output directory, default a new temporary directory]
cd "$(dirname "$0")/../.."
OUT="${1:-$(mktemp -d)}"
echo "outputs: $OUT"
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/as_gpu.txt"
python -c "import __graft_entry__ as g; g.build()" || exit 1
timeout 1200 python -m pytest tests/test_dfpn_amp.py -q -m gpu -rs 2>&1 | grep -v "^\.*$" | tail -40 | tee "$OUT/as_amp_tests.txt"
timeout 1800 python -m pytest tests -q -m gpu 2>&1 | tail -6 | tee "$OUT/as_gputest.txt"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
timeout 300 python bench.py --gpus 1 --steps 50 --warmup 5 > "$OUT/as_bench_align.json" 2>/dev/null; tail -c 400 "$OUT/as_bench_align.json"
timeout 900 python tools/gpu/time_dfpn_amp.py "$OUT/as_time_dfpn_amp.json" 2>&1 | tail -16
