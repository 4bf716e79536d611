#!/bin/bash
# One run on the GPU: the decode on float32 / bfloat16 / float16 maps and on float16 maps up-cast by the caller (K1, grouping,
# whole call), config 5 with a bf16 and a float16 network, and decode_host_batch by input dtype. Arms alternate, rounds
# repeat; the card's name, power limit and clocks are recorded in the same run.
# usage: bash tools/gpu_dtypes.sh <output directory> [rounds]
out=${1:?usage: bash tools/gpu_dtypes.sh <output directory> [rounds]}
rounds=${2:-2}
mkdir -p $out
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv > $out/gpu.txt 2>&1; nproc >> $out/gpu.txt
for r in $(seq 1 $rounds); do
  for dt in bf16 f16 upcast f32; do
    timeout 200 python tools/bench_k1.py 180x320 4096 10 $dt >> $out/bench_k1.log 2>&1
    timeout 200 python tools/bench_k1.py 64x64 32768 10 $dt lean >> $out/bench_k1.log 2>&1
  done
done
grep -v Warn $out/bench_k1.log
for dt in bf16 f16; do
  timeout 300 python tools/bench_config5.py 256 5 $dt >> $out/config5.jsonl 2> $out/config5_$dt.err
done
cat $out/config5.jsonl
timeout 600 python tools/bench_host_dtypes.py 2048 5 3 > $out/host_dtypes.json 2> $out/host_dtypes.err; cat $out/host_dtypes.json
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks_throttle_reasons.active --format=csv >> $out/gpu.txt 2>&1
