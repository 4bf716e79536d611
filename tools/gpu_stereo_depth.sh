#!/bin/bash
# One run on the GPU: the depth-association tests, the stereo-objects tests, then tools/bench_stereo.py (both association
# modes timed in the same rounds, and the same-row accuracy lines); the card's name, power limit and clocks in the same run.
# usage: bash tools/gpu_stereo_depth.sh <output directory> [rounds]
out=${1:?usage: bash tools/gpu_stereo_depth.sh <output directory> [rounds]}
rounds=${2:-5}
mkdir -p $out
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv > $out/gpu.txt 2>&1
timeout 1500 python -m pytest -q -s -p no:cacheprovider tests/test_gpu_stereo_depth.py tests/test_gpu_stereo_objects.py > $out/tests.txt 2>&1
echo "tests exit $?" >> $out/tests.txt
timeout 900 python tools/bench_stereo.py $rounds > $out/stereo.txt 2> $out/stereo.err
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks_throttle_reasons.active --format=csv >> $out/gpu.txt 2>&1
tail -3 $out/tests.txt
cat $out/gpu.txt $out/stereo.txt
