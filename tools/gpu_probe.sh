#!/bin/bash
# First-contact probe of the fused kernel on a B200: each case runs in its own process under `timeout`.
mkdir -p gpurun_out
LOG=gpurun_out/probe.log
: > $LOG
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv >> $LOG 2>&1
for C in "256 1000 512 1" "7 300 100 3" "130 257 384 2" "513 4097 512 5" "300 20000 512 10" "2000 3000 256 16" "10000 100000 512 1" "10000 100000 512 10"; do
  echo "== case $C" >> $LOG
  timeout 120 python tools/gpu_case.py $C >> $LOG 2>&1
  echo "exit=$?" >> $LOG
done
tail -60 $LOG
