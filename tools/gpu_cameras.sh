#!/bin/bash
# One run on the GPU: tools/bench_cameras.py (one camera per call, camera tables with one and two cameras, a stereo batch
# split into two calls) at 180x320 and 64x64 (lean tables); the card's name, power limit and clocks in the same run.
# usage: bash tools/gpu_cameras.sh <output directory> [rounds]
out=${1:?usage: bash tools/gpu_cameras.sh <output directory> [rounds]}
rounds=${2:-3}
mkdir -p $out
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv > $out/gpu.txt 2>&1
timeout 600 python tools/bench_cameras.py 180x320 4096 10 $rounds > $out/cameras_180x320.txt 2> $out/cameras_180x320.err
timeout 600 python tools/bench_cameras.py 64x64 32768 10 $rounds lean > $out/cameras_64x64.txt 2> $out/cameras_64x64.err
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks_throttle_reasons.active --format=csv >> $out/gpu.txt 2>&1
cat $out/gpu.txt $out/cameras_180x320.txt $out/cameras_64x64.txt
