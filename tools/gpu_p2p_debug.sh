#!/bin/bash
OUT=gpurun_out; mkdir -p $OUT
echo "== tests"; timeout 600 python -m pytest tests/test_distributed_gpu.py -q --timeout=500 2>&1 | tail -3
run() { python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29517 bench.py --gpus 2 --steps 20 --warmup 3 --no-qv 2>/dev/null | python -c "
import sys,json
d=json.loads([l for l in sys.stdin if l.startswith('{')][-1]); print('$1', 'ms/step',round(d['ms_per_step'],3),'fused launch us', round(d['roofline']['launch_ms']*1e3,1))"; }
PP2D_P2P=0 run nccl
PP2D_P2P_DEBUG=7 run p2p_nothing
PP2D_P2P_DEBUG=5 run p2p_stores_only
PP2D_P2P_DEBUG=0 run p2p_full
