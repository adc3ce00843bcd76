#!/bin/bash
# Multi-GPU session: sharded-solve parity tests (spawn, p2p transport) and the bench at N ranks.  usage: scripts/gpu_r2_multi.sh <tag> <N>
set -u
T=${1:-r2m}
N=${2:-2}
O=gpurun_out
mkdir -p $O
nvidia-smi --query-gpu=index,name --format=csv > $O/${T}_smi.txt 2>&1
nvidia-smi topo -m >> $O/${T}_smi.txt 2>&1
timeout 900 python -m pytest tests/test_ba_multigpu.py -m gpu -q --durations=10 > $O/${T}_pytest.log 2>&1; echo "pytest rc=$?" >> $O/${T}_pytest.log
timeout 600 python bench.py --gpus 1 --steps 8 --warmup 3 --no-detect --no-clahe --no-marg --no-keyframe --no-cpu-baseline > $O/${T}_bench1.json 2> $O/${T}_bench1.err; echo "bench1 rc=$?" >> $O/${T}_bench1.err
timeout 900 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29531 bench.py --gpus $N --steps 8 --warmup 3 \
    --no-detect --no-clahe --no-marg --no-keyframe > $O/${T}_bench${N}.json 2> $O/${T}_bench${N}.err; echo "bench rc=$?" >> $O/${T}_bench${N}.err
tail -12 $O/${T}_pytest.log; python - <<PY
import json
for n in (1, $N):
    try:
        d = json.loads(open("$O/${T}_bench%d.json" % n).read().strip().splitlines()[-1])
        print("N", d["n_gpus"], "value", round(d["value"]), "e2e", round(d["e2e"]["value"]), "sharded", {k: v for k, v in d["sharded_ba"].items() if k != "workload"})
    except Exception as e:
        print("bench parse failed", n, e)
PY
tail -5 $O/${T}_bench${N}.err
