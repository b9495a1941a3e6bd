#!/bin/bash
# round-end measurement suite (one gpurun call): tests, bench lines, ncu launch list, one ncu --set full capture
set -x
O=gpurun_out
timeout 900 python -m pytest tests -m gpu -q 2>&1 | tail -3
python bench.py > $O/bench_cfg2.json 2> $O/bench_cfg2.err
for wl in cfg1 cfg3 cfg4 cfg5; do python bench.py --workload $wl > $O/bench_$wl.json 2>/dev/null; done
python bench.py --impl reference --steps 3 --warmup 1 > $O/bench_reference.json 2>/dev/null
CMD="python bench.py --steps 20 --warmup 3 --no-cpu-baseline --e2e-steps 1"
$CMD > $O/plain.log 2>&1 &&
ncu --metrics gpu__time_duration.sum --clock-control none -s 40 -c 50 --csv --log-file $O/launches_cfg2.csv $CMD > $O/ncu_l.log 2>&1
$CMD > $O/plain.log 2>&1 &&
ncu --set full --clock-control none --import-source on -k regex:"warp_staged|cm_" -s 25 -c 5 -f -o $O/prof_cfg2 $CMD > $O/ncu_f.log 2>&1
bash profiles/r1_sweep_cm2.sh
