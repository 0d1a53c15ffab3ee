#!/bin/bash
# usage (on an N-GPU box): tools/scale_artifacts.sh r02 [N]   -- host copy ceiling for 1/2/4/8 busy GPUs, bench lines at 2/4/8 ranks
# (config 3, strong scaling), and the multi-device tests.
tag=${1:-r02}; N=${2:-8}
timeout 200 python tools/pcie_probe_multi.py $N > gpurun_out/${tag}_pcie_probe_multi.txt 2>&1; tail -4 gpurun_out/${tag}_pcie_probe_multi.txt
timeout 200 python -m pytest tests/test_gpu_parity.py -q -k "two_devices or all_devices" > gpurun_out/t_${tag}_multidev.log 2>&1; tail -2 gpurun_out/t_${tag}_multidev.log
for n in $N 4 2; do
  [ $n -le $N ] || continue
  timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node $n --master-addr 127.0.0.1 --master-port 2951$n bench.py --gpus $n --steps 5 --warmup 2 > gpurun_out/bench_${tag}_n$n.log 2>&1
  tail -1 gpurun_out/bench_${tag}_n$n.log > gpurun_out/${tag}_bench_line_n$n.json; cut -c1-300 gpurun_out/${tag}_bench_line_n$n.json
done
nvidia-smi topo -m > gpurun_out/${tag}_topo.txt 2>&1; lscpu | grep -E "Model name|Socket|NUMA|^CPU\(s\)" >> gpurun_out/${tag}_topo.txt
