#!/bin/bash
# Round-2 single-GPU session I: split-pipeline tests, cfg-4 stage profile + phase clocks, full GPU suite, short bench.
set -u
T=${1:-r2i}
O=gpurun_out
mkdir -p $O
timeout 600 python -m pytest tests/test_ba_gpu.py -q -m gpu -x -k "cfg4 or sharded" > $O/${T}_pytest_split.log 2>&1; echo "pytest split rc=$?" | tee -a $O/${T}_pytest_split.log
tail -5 $O/${T}_pytest_split.log
ICG_BA_PROFILE=1 timeout 200 python scripts/prof_ba.py 32 3 20 2000 > $O/${T}_ba_stages_cfg4.log 2>&1
ICG_LIB_VARIANT=prof ICG_BA_PROFILE=1 timeout 200 python scripts/prof_ba.py 32 3 20 2000 > $O/${T}_ba_phase_clocks_cfg4.log 2>&1
tail -22 $O/${T}_ba_stages_cfg4.log; sed -n '/ba_solve_cam_dsm phases/,$p' $O/${T}_ba_phase_clocks_cfg4.log
timeout 900 python -m pytest tests -q -m gpu > $O/${T}_pytest.log 2>&1; echo "pytest rc=$?" | tee -a $O/${T}_pytest.log
tail -4 $O/${T}_pytest.log
timeout 200 python __graft_entry__.py --smoke > $O/${T}_smoke.log 2>&1; echo "smoke rc=$?" | tee -a $O/${T}_smoke.log
timeout 400 python bench.py --no-cpu-baseline --no-marg --no-detect --no-clahe --no-keyframe > $O/${T}_bench.json 2> $O/${T}_bench.err; echo "bench rc=$?"
python - <<PY
import json
d=json.loads(open('$O/${T}_bench.json').read().strip().splitlines()[-1])
print('value',round(d['value']),'ms/step',d['ms_per_step'],'e2e',round(d['e2e']['value']),'ba_only',d.get('ba_only',{}).get('solves_per_s'))
print('sharded',{k:v for k,v in d.get('sharded_ba',{}).items() if k!='workload'})
PY
