#!/bin/bash
# CUDA start-up probe: one process / N concurrent processes, one visible device each or all, with a 1 TB arena, with busy CPUs.
mkdir -p gpurun_out
N=${1:-2}
P=scripts/probe/ctx_probe
[ -x $P ] || nvcc -gencode arch=compute_100a,code=sm_100a -O2 -std=c++17 -o $P $P.cu -lcuda || exit 1
nproc; nvidia-smi --query-gpu=persistence_mode --format=csv,noheader | head -1
{
echo "== single process, one device (x3)"; for i in 1 2 3; do CUDA_VISIBLE_DEVICES=0 $P -tag single; done
echo "== single process, all $N devices"; $P -tag all
echo "== single, one device, 1 TB arena"; CUDA_VISIBLE_DEVICES=0 $P -arena 1024 -tag arena
echo "== single, one device, 16 busy threads"; CUDA_VISIBLE_DEVICES=0 $P -busy 16 -tag busy16
echo "== $N concurrent processes, one device each"; for g in $(seq 0 $((N-1))); do CUDA_VISIBLE_DEVICES=$g $P -tag conc$g & done; wait
echo "== again"; for g in $(seq 0 $((N-1))); do CUDA_VISIBLE_DEVICES=$g $P -tag conc$g & done; wait
echo "== $N processes staggered by 0.3 s"; for g in $(seq 0 $((N-1))); do CUDA_VISIBLE_DEVICES=$g $P -tag stag$g & sleep 0.3; done; wait
echo "== 2 concurrent processes on the SAME device"; for g in 0 1; do CUDA_VISIBLE_DEVICES=0 $P -tag same$g & done; wait
} 2>&1 | tee gpurun_out/r2_ctx_probe_n$N.txt
