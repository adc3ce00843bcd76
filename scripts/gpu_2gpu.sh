#!/bin/bash
# 2-GPU checks: landmark-sharded solve parity vs the oracle (cfg 3 and cfg 4) + the scaling bench at N = 2
T=${1:-g2}
O=gpurun_out
mkdir -p $O
timeout 700 python -m pytest tests/test_ba_multigpu.py -q -m gpu > $O/${T}_shard.log 2>&1
timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29513 bench.py --gpus 2 --steps 6 --warmup 3 > $O/${T}_bench2.json 2> $O/${T}_bench2.err
tail -4 $O/${T}_shard.log; tail -c 1500 $O/${T}_bench2.json; tail -3 $O/${T}_bench2.err
