#!/bin/bash
# 2 GPUs: the sharded solve (NCCL all-reduce of the LM try) against the single-GPU solve, and cfg 3 on 2 GPUs
cd "${GRAFT_REPO_ROOT:-.}"; mkdir -p gpurun_out
export AAR_RIG_CACHE=/tmp/rigs
timeout 300 python -m pytest tests/test_gpu_multi.py -x -q -m gpu -s -k "world2 or 2" > gpurun_out/multi_n2_pytest_multi.txt 2>&1; tail -6 gpurun_out/multi_n2_pytest_multi.txt | cut -c1-600
run() { n=$1; shift; timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node $n --master-addr 127.0.0.1 --master-port 29512 bench.py --gpus $n "$@"; }
run 2 --workload cfg3 --steps 20 --warmup 3 2>/dev/null | python -c "
import json,sys
d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print('cfg3 n2 nccl', d['ms_per_step'], d['e2e']['ms_per_step'])"
