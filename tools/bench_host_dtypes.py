"""decode_host_batch throughput by input dtype: pinned 180x320 valve frames (bench.py's seed 1004) in, pinned tables out,
128-frame chunks. Four arms, run in alternation (round r times every arm once, in a rotated order) so that drift of a
shared host hits all of them alike:
  f32_auto   float32, sparse='auto' (the host pass marks tiles; dense copies side by side)
  f32_dense  float32, sparse=False (every heatmap byte crosses PCIe)
  bf16       bfloat16 (16-bit maps always cross densely: half the bytes)
  f16        float16
Depth and centre maps are pinned, so they are gathered in place in every arm. Prints one JSON line: the median
frames/s of each arm over the rounds, the bytes each step sent over PCIe, and whether each arm's tables equal those of
decode_batch on the same maps on the device.
usage: python tools/bench_host_dtypes.py [frames] [rounds] [steps]"""
import json
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from object_keypoints_b200 import KeypointDecoder, synthetic

frames = int(sys.argv[1]) if len(sys.argv) > 1 else 2048
rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 5
steps = int(sys.argv[3]) if len(sys.argv) > 3 else 3
cfg, size = [1, 3], (180, 320)
maps = synthetic.torch_grid_batch(frames, cfg, size, seed=1004, grid=(4, 2), device='cuda')[:3]
decoder = KeypointDecoder(cfg, size, camera=synthetic.default_camera(size))
arms = {'f32_auto': (torch.float32, 'auto'), 'f32_dense': (torch.float32, False),
        'bf16': (torch.bfloat16, 'auto'), 'f16': (torch.float16, 'auto')}
host = {dtype: [t.to(dtype).cpu().pin_memory() for t in maps] for dtype in {d for d, _ in arms.values()}}
outs, rates, sent, parity = {}, {name: [] for name in arms}, {}, {}


def run(name):
    dtype, sparse = arms[name]
    outs[name] = decoder.decode_host_batch(*host[dtype], chunk_frames=128, sparse=sparse, out=outs.get(name))
    return decoder.host_bytes_copied


for name, (dtype, _) in arms.items():                   # warm-up (staging buffers, the pack worker) + parity
    run(name)
    sent[name] = run(name)
    want = decoder.decode_batch(*(t.to(dtype) for t in maps)).numpy()
    parity[name] = all(np.array_equal(outs[name][k].numpy().view(np.uint8), want[k].view(np.uint8))
                       for k in KeypointDecoder.HOST_RESULT_TABLES)
names = list(arms)
for r in range(rounds):
    for name in names[r % len(names):] + names[:r % len(names)]:
        torch.cuda.synchronize()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for _ in range(steps):
            run(name)                                   # returns after its own synchronise
        stop.record()
        stop.synchronize()
        rates[name].append(frames * steps / (start.elapsed_time(stop) / 1e3))
print(json.dumps({'workload': f'decode_host_batch, {frames} pinned frames of 180x320, chunks of 128', 'rounds': rounds,
                  'steps_per_round': steps, 'host_threads': os.cpu_count(),
                  'frames_per_s_median': {k: float(np.median(v)) for k, v in rates.items()},
                  'frames_per_s_min_max': {k: [min(v), max(v)] for k, v in rates.items()},
                  'h2d_bytes_per_step': sent, 'tables_equal_device_decode': parity}))
