#!/bin/bash
# Round 2, multi-GPU call (run under `gpurun --gpus N`, N = 2 first, then 8): the peer-memory all-reduce's first
# multi-process run against NCCL, then weak and strong scaling with whichever is the default.
#   gpurun --gpus 2 --timeout 900 -- bash scripts/gpu_run_round2_scaling.sh 2
#   gpurun --gpus 8 --timeout 1500 -- bash scripts/gpu_run_round2_scaling.sh 8
N=${1:-2}
mkdir -p gpurun_out
nvidia-smi topo -m > gpurun_out/r2_topo$N.txt 2>&1
PORT=29600
run() {   # tag, env assignments, bench arguments
  local tag=$1 envs=$2; shift 2
  PORT=$((PORT+1))
  env $envs timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port $PORT \
      bench.py --gpus $N --steps 20 --warmup 5 --no-e2e "$@" > gpurun_out/r2_n${N}_$tag.json 2> gpurun_out/r2_n${N}_$tag.err
  echo "$tag exit $?" >> gpurun_out/r2_n${N}_$tag.err
  echo "== $tag"; python scripts/show_bench.py gpurun_out/r2_n${N}_$tag.json 2>/dev/null | head -3; tail -2 gpurun_out/r2_n${N}_$tag.err | cut -c1-300
}
run weak_nccl  "AECF_DP_COLLECTIVE=nccl"
run weak_peer  "AECF_DP_COLLECTIVE=peer"
run strong_nccl "AECF_DP_COLLECTIVE=nccl" --global-batch 65536
run strong_peer "AECF_DP_COLLECTIVE=peer" --global-batch 65536
timeout 200 python bench.py --gpus 1 --steps 20 --warmup 5 --no-cpu-baseline --no-e2e > gpurun_out/r2_n${N}_same_box_n1.json 2> gpurun_out/r2_n${N}_same_box_n1.err
echo "== n1 on the same box"; python scripts/show_bench.py gpurun_out/r2_n${N}_same_box_n1.json 2>/dev/null | head -2
