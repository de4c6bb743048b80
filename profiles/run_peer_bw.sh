#!/bin/bash
# gpurun --gpus 2 --timeout 600 -- 'bash profiles/run_peer_bw.sh r02j 2'
R=${1:-r02j}; N=${2:-2}
mkdir -p gpurun_out
timeout 200 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 \
      --master-port 29511 profiles/peer_bw.py 2>/dev/null | grep '^{' >> gpurun_out/${R}_peer_bw_n$N.jsonl
cat gpurun_out/${R}_peer_bw_n$N.jsonl
