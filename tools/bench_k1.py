"""Times okp_extract_peaks_* (K1) and okp_group_objects_* alone, and the fused okp_decode_* call, on synthetic batches.
usage: python tools/bench_k1.py [180x320|64x64] [frames] [reps] [f32|bf16] [lean]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from object_keypoints_b200 import KeypointDecoder, synthetic

shape = sys.argv[1] if len(sys.argv) > 1 else '180x320'
frames = int(sys.argv[2]) if len(sys.argv) > 2 else 2048
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 10
dtype = sys.argv[4] if len(sys.argv) > 4 else 'f32'
H, W = [int(v) for v in shape.split('x')]
grid = (4, 2) if W >= 128 else (2, 1)
heat, depth, centers, _ = synthetic.torch_grid_batch(frames, [1, 3], (H, W), seed=7, grid=grid, device='cuda')
if dtype == 'bf16':
    heat, depth, centers = heat.bfloat16(), depth.bfloat16(), centers.bfloat16()
camera = synthetic.default_camera((H, W))
flags = sys.argv[5:]
lean = 'lean' in flags
if 'nocam' in flags:
    camera = None                      # grouping without the 3D lift (isolates the float64 Newton / tan chains)
dec = KeypointDecoder([1, 3], (H, W), camera=camera, lean_tables=lean, single_pass='single' in flags)
tables = dec.tables(frames)
ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
k1 = k3 = 0.0
for _ in range(0 if 'fusedonly' in flags else 3):
    dec.extract_peaks(heat, tables); dec.group_objects(depth, centers, tables)
torch.cuda.synchronize()
for _ in range(0 if 'fusedonly' in flags else reps):
    ev[0].record(); dec.extract_peaks(heat, tables); ev[1].record(); dec.group_objects(depth, centers, tables); ev[2].record()
    torch.cuda.synchronize()
    k1 += ev[0].elapsed_time(ev[1]); k3 += ev[1].elapsed_time(ev[2])
k1 = max(k1 / reps, 1e-9); k3 /= reps
for _ in range(3):
    dec.decode_batch(heat, depth, centers, tables=tables)
torch.cuda.synchronize()
ev[0].record()
for _ in range(reps):
    dec.decode_batch(heat, depth, centers, tables=tables)
ev[1].record()
torch.cuda.synchronize()
fused = ev[0].elapsed_time(ev[1]) / reps
gb = frames * 3 * H * W * heat.element_size() / 1e9
print(f"{shape} {dtype} frames={frames} "
      f"K1 {k1 * 1e3:.1f} us = {gb / (k1 / 1e3):.0f} GB/s ({gb / (k1 / 1e3) / 6547.2:.3f} of measured HBM peak); group {k3 * 1e3:.1f} us; "
      f"decode_batch {' '.join(flags)} {fused * 1e3:.1f} us = {gb / (fused / 1e3) / 6547.2:.3f}; "
      f"objects/frame {float(tables['n_objects'].float().mean()):.2f}")
