#!/bin/bash
# One run on the GPU: the sequence-objects tests and the existing sequence tests, then tools/bench_sequence_objects.py
# (decode, per-peak chain and both association modes of the object chain timed in the same rounds, and the accuracy
# lines); the card's name, power limit and clocks in the same run.
# usage: bash tools/gpu_sequence_objects.sh <output directory> [rounds]
out=${1:?usage: bash tools/gpu_sequence_objects.sh <output directory> [rounds]}
rounds=${2:-5}
mkdir -p $out
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv > $out/gpu.txt 2>&1
timeout 1500 python -m pytest -q -s -p no:cacheprovider tests/test_gpu_sequence_objects.py tests/test_sequence.py > $out/tests.txt 2>&1
echo "tests exit $?" >> $out/tests.txt
timeout 900 python tools/bench_sequence_objects.py $rounds > $out/sequence.txt 2> $out/sequence.err
echo "bench exit $?" >> $out/sequence.txt
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks_throttle_reasons.active --format=csv >> $out/gpu.txt 2>&1
tail -3 $out/tests.txt
cat $out/gpu.txt $out/sequence.txt
tail -5 $out/sequence.err
