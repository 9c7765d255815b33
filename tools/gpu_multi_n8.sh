#!/bin/bash
# 8 GPUs of one box: multi-GPU parity (world 2 and 8), cfg 4 at N = 8 with NCCL all-reduces
cd "${GRAFT_REPO_ROOT:-.}"; mkdir -p gpurun_out
export AAR_RIG_CACHE=/tmp/rigs
timeout 600 python -m pytest tests/test_gpu_multi.py -x -q -m gpu -s > gpurun_out/multi_n8_pytest_multi.txt 2>&1; tail -3 gpurun_out/multi_n8_pytest_multi.txt | cut -c1-700
python - <<'PY'
import sys, time
sys.path.insert(0, "automatic-ar_b200/python")
from aar_b200 import synth
t = time.time(); synth.make_config("cfg4"); print("rig cached", time.time() - t)
PY
run() { n=$1; shift; timeout 400 python -m torch.distributed.run --nnodes=1 --nproc-per-node $n --master-addr 127.0.0.1 --master-port 29513 bench.py --gpus $n "$@"; }
run 8 --steps 20 --warmup 3 > gpurun_out/multi_n8_bench_cfg4_n8_nccl.json 2> gpurun_out/multi_n8_bench_cfg4_n8_nccl.err; python - <<'PY'
import json
try:
    d=json.loads(open("gpurun_out/multi_n8_bench_cfg4_n8_nccl.json").read().strip().splitlines()[-1]); print("cfg4 n8 nccl", d["ms_per_step"], d["e2e"]["ms_per_step"], d["config"]["lm_loop"], "final cost", d["final_cost"])
except Exception as e: print("parse failed", e)
PY
