#!/bin/bash
# run dist_gpu_worker with all ranks on cuda:0 (gloo); $1 = ranks, extra env via environment
cd /root/repo
port=$((20000 + RANDOM % 20000))
for r in $(seq 0 $(($1 - 1))); do
  RANK=$r WORLD_SIZE=$1 LOCAL_RANK=0 MASTER_ADDR=127.0.0.1 MASTER_PORT=$port SB200_TEST_SINGLE_DEVICE=1 SB200_PEER_WAIT_S=${SB200_PEER_WAIT_S:-60} \
    python tests/dist_gpu_worker.py > gpurun_out/sd_$r.log 2>&1 &
done
wait
for r in $(seq 0 $(($1 - 1))); do echo "--- rank $r"; grep -v "WARNING\|^$\|=====\|resolved\|grid of" gpurun_out/sd_$r.log | tail -6; done
