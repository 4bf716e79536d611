"""BASELINE config 5: random-init CornerNet-Squeeze forward at batch 256 feeding the decode kernels.
The network is the input producer (plain PyTorch / cuDNN, not the product); its three head outputs stay
on the device and go straight into okp_decode_bf16 (or okp_decode_f16 for a float16 network).
Reports end-to-end frames/s and the decode share.
usage: python tools/bench_config5.py [batch] [reps] [bf16|f16]"""
import json
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from object_keypoints_b200 import KeypointDecoder, producer, synthetic

batch = int(sys.argv[1]) if len(sys.argv) > 1 else 256
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
kind = sys.argv[3] if len(sys.argv) > 3 else 'bf16'
dtype = {'bf16': torch.bfloat16, 'f16': torch.float16}[kind]
cfg = [1, 3]
torch.backends.cudnn.benchmark = True
net = producer.build_producer(cfg, device='cuda', dtype=dtype, seed=0)
torch.manual_seed(0)
frames = torch.randn(batch, 3, 511, 511, device='cuda', dtype=dtype).contiguous(memory_format=torch.channels_last)
camera = synthetic.default_camera((64, 64))
# random-init heatmaps sit at ~0.5 everywhere: ~100 noise peaks per map (SURVEY.md 8d #5) -> large tables
decoder = KeypointDecoder(cfg, (64, 64), camera=camera, max_peaks=128, max_objects=128, max_votes=64)
tables = decoder.tables(batch)
ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
with torch.no_grad():
    for _ in range(3):
        heat, depth, centers = net(frames)
        decoder.decode_batch(heat, depth, centers, tables=tables)
    torch.cuda.synchronize()
    t_net = t_dec = 0.0
    for _ in range(reps):
        ev[0].record()
        heat, depth, centers = net(frames)
        ev[1].record()
        decoder.decode_batch(heat, depth, centers, tables=tables)
        ev[2].record()
        torch.cuda.synchronize()
        t_net += ev[0].elapsed_time(ev[1]); t_dec += ev[1].elapsed_time(ev[2])
t_net /= reps; t_dec /= reps
peaks = tables['peak_count'].float().mean().item()
print(json.dumps({'workload': f'config5: CornerNet-Squeeze {kind} forward -> okp_decode_{kind}', 'batch': batch, 'reps': reps,
                  'network_ms': t_net, 'decode_ms': t_dec, 'frames_per_s': batch / ((t_net + t_dec) / 1e3),
                  'decode_share': t_dec / (t_net + t_dec), 'mean_peaks_per_map': peaks,
                  'overflow_frames': int((tables['flags'] & 1).ne(0).sum().item()), 'dtype': kind,
                  'data': 'synthetic randn frames, random-init weights'}))
