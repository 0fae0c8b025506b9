#!/bin/bash
# round-2 multi-GPU call: host link probe, the 1->8 curve points, configs[4] on N GPUs
N=${1:-8}
TR="python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1"
mkdir -p gpurun_out/s$N
nvidia-smi topo -m > gpurun_out/s$N/topo.txt 2>&1
lscpu | head -25 > gpurun_out/s$N/lscpu.txt 2>&1
$TR --master-port 29601 tools/pcie_probe.py > gpurun_out/s$N/pcie_probe.txt 2>&1; tail -3 gpurun_out/s$N/pcie_probe.txt
$TR --master-port 29602 bench.py --gpus $N --steps 10 --warmup 3 > gpurun_out/s$N/bench.json 2> gpurun_out/s$N/bench.err
grep '^{' gpurun_out/s$N/bench.json | python -c "import json,sys; d=json.loads(sys.stdin.read()); print('bench', d['n_gpus'], d['value'], d['ms_per_step'], 'e2e', d['e2e']['value'], d['e2e']['ms_per_step'], d['kernel_ms'])"
$TR --master-port 29604 tools/stress_bench.py --frames 1025 --steps 3 2>&1 | grep '^{' > gpurun_out/s$N/stress.json; cut -c1-900 gpurun_out/s$N/stress.json
