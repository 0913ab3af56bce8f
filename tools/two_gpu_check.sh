#!/bin/bash
# two GPUs of one box: one host thread driving two devices; the bench under torchrun with one sequence per GPU
cd "$GRAFT_REPO_ROOT"
mkdir -p gpurun_out
nvidia-smi -L | head -4
timeout 200 python -m pytest tests/test_gpu_parity.py -m gpu -x -q -p no:cacheprovider -k "two_devices" 2>&1 | tail -2
timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 bench.py --gpus 2 --steps 20 --warmup 5 --no-nn --no-cpu --no-extra --streams 0 > gpurun_out/r2_bench_2gpus.json 2> gpurun_out/r2_bench_2gpus.err
echo "bench2 rc=$?"; python -c "
import json; d=json.loads(open('gpurun_out/r2_bench_2gpus.json').read().strip().splitlines()[-1])
print('n_gpus', d['n_gpus'], 'value', d['value'], 'e2e', d['e2e']['value'], 'per-rank ms per scan', d['windows']['value']['median_ms_per_scan_per_rank'])"
