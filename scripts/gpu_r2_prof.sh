#!/bin/bash
# Round-2 profiling session (one GPU): KLT A/B (4 vs 5 resident CTAs), BA stage timings (fused cfg 3, split cfg 4),
# ncu launch list of the bench command, ncu --set full of the KLT tracker and of the cluster solve.   usage: scripts/gpu_r2_prof.sh <tag>
set -u
T=${1:-r2p}
O=gpurun_out
mkdir -p $O
for MB in 4 5; do
  ICG_KLT_MINB=$MB timeout 300 python bench.py --steps 10 --warmup 3 --no-ba --no-cpu-baseline --no-detect --no-clahe --no-sharded --no-marg --no-keyframe > $O/${T}_klt_minb$MB.json 2> $O/${T}_klt_minb$MB.err
done
ICG_BA_PROFILE=1 timeout 300 python scripts/prof_ba.py 148 4 > $O/${T}_ba_stages_cfg3.log 2>&1
ICG_BA_PROFILE=1 timeout 300 python scripts/prof_ba.py 32 3 20 2000 > $O/${T}_ba_stages_cfg4.log 2>&1
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 2500 --csv --log-file $O/${T}_launches.csv \
   python bench.py --steps 2 --warmup 1 --streams 148 --no-cpu-baseline --no-sharded --no-marg --no-detect --no-clahe --no-keyframe > $O/${T}_ncu_bench.log 2>&1
timeout 600 ncu --set full --clock-control none --import-source on -k regex:klt_track -s 1 -c 1 -f -o $O/${T}_klt_track \
   python bench.py --steps 1 --warmup 1 --streams 148 --no-cpu-baseline --no-sharded --no-ba --no-detect --no-clahe --no-keyframe > $O/${T}_ncu_klt.log 2>&1
timeout 600 ncu --set full --clock-control none --import-source on -k regex:ba_solve_cam -s 3 -c 1 -f -o $O/${T}_solve_cam \
   python scripts/prof_ba.py 8 1 20 2000 > $O/${T}_ncu_solve_cam.log 2>&1
timeout 300 python scripts/prof_marg.py 148 3 > $O/${T}_marg.log 2>&1
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file $O/${T}_marg_launches.csv python scripts/prof_marg.py 148 1 > $O/${T}_ncu_marg.log 2>&1
for f in $O/${T}_klt_minb4.json $O/${T}_klt_minb5.json; do python -c "
import json,sys
d=json.loads(open('$f').read().strip().splitlines()[-1]); print('$f', round(d['value']), d['roofline']['kernel_ms'], round(d['roofline']['frac'],4))"; done
cat $O/${T}_marg.log; python scripts/launch_summary.py $O/${T}_marg_launches.csv 2>/dev/null | head -20; tail -14 $O/${T}_ba_stages_cfg3.log; tail -16 $O/${T}_ba_stages_cfg4.log
