#!/bin/bash
# cfg 3 (8 cameras, 24 markers, 10 k frames) sharded over the GPUs of this box; on 2 GPUs also the multi-GPU parity test
cd "${GRAFT_REPO_ROOT:-.}"; mkdir -p gpurun_out
export AAR_RIG_CACHE=/tmp/rigs
N=$(nvidia-smi -L | wc -l)
if [ $N -eq 2 ]; then timeout 300 python -m pytest tests/test_gpu_multi.py -x -q -m gpu > gpurun_out/cfg3_pytest_multi_n2.txt 2>&1; tail -2 gpurun_out/cfg3_pytest_multi_n2.txt; fi
timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29514 bench.py --gpus $N --workload cfg3 --steps 20 --warmup 3 > gpurun_out/cfg3_bench_cfg3_n$N.json 2> gpurun_out/cfg3_bench_cfg3_n$N.err
python - <<PY
import json
d=json.loads(open("gpurun_out/cfg3_bench_cfg3_n$N.json").read().strip().splitlines()[-1]); print("cfg3 n$N", d["ms_per_step"], d["e2e"]["ms_per_step"], d["config"]["lm_loop"], d["final_cost"])
PY
