#!/bin/bash
# Final multi-GPU check: sharded-vs-single cases, headline bench.
set -x
N=${1:-2}
mkdir -p gpurun_out
BLADES_MGPU_SIZES=1,$N timeout 900 python -m pytest tests/test_multigpu.py -m gpu -q --timeout 600 -k "dead_rank or trimmedmean-alie-mlp or krum-noise or geomed or resnet18" > gpurun_out/pytest_multigpu_final_$N.log 2>&1; echo "exit $?"; tail -12 gpurun_out/pytest_multigpu_final_$N.log | cut -c1-300
timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29555 bench.py --gpus $N --steps 30 --warmup 5 --no-port > gpurun_out/bench_${N}gpu_final.json 2> gpurun_out/bench_${N}gpu_final.err
tail -1 gpurun_out/bench_${N}gpu_final.json | cut -c1-200; tail -1 gpurun_out/bench_${N}gpu_final.json | grep -o '"e2e".\{0,200\}'; grep -v "OMP\|\*\*\*" gpurun_out/bench_${N}gpu_final.err | tail -3 | cut -c1-300
