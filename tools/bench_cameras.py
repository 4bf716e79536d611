"""Per-frame cameras against one camera per call, CUDA events. Four arms on the same float32 maps:
  reset   one camera for the batch (KeypointDecoder.reset: okp_decode_emit_f32 / okp_group_objects_emit_f32)
  table1  a camera table holding that camera on every row (okp_decode_cameras_f32 / okp_group_objects_cameras_f32)
  table2  a camera table with cam0 / cam1 alternating (a stereo batch, left and right views interleaved)
  split   what a stereo caller does without the table: two calls of N/2 frames, one per camera
For each arm: K1 (okp_extract_peaks_f32), the grouping kernel and the whole decode call, in us per batch. Arms alternate
within a round; rounds repeat. The maps are ~2.8 GB (180x320) / ~1.6 GB (64x64): larger than L2.
usage: python tools/bench_cameras.py [180x320|64x64] [frames] [reps] [rounds] [lean]"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from object_keypoints_b200 import KeypointDecoder, camera_utils, synthetic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
shape = sys.argv[1] if len(sys.argv) > 1 else '180x320'
frames = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 10
rounds = int(sys.argv[4]) if len(sys.argv) > 4 else 2
lean = 'lean' in sys.argv[5:]
H, W = [int(v) for v in shape.split('x')]
cfg = [1, 3]
heat, depth, centers, _ = synthetic.torch_grid_batch(frames, cfg, (H, W), seed=7, grid=(4, 2) if W >= 128 else (2, 1),
                                                     device='cuda')
half = frames // 2

params = camera_utils.load_calibration_params(os.path.join(ROOT, 'config', 'calibration.yaml'))
rig = [camera_utils.FisheyeCamera(params[k], params[d], params['image_size']) for k, d in (('K', 'D'), ('Kp', 'Dp'))]
if (H, W) == (64, 64):
    def fit(camera):
        scaled = camera.scale(511.0 / 720.0)
        return scaled.cut(np.array([(scaled.image_size[1] - 511.0) / 2.0, 0.0])).scale(64.0 / 511.0)
else:
    def fit(camera):
        return camera.scale(H / 720.0)
cam0, cam1 = (fit(c) for c in rig)

decoder = KeypointDecoder(cfg, (H, W), camera=cam0, lean_tables=lean)
split = [KeypointDecoder(cfg, (H, W), camera=c, lean_tables=lean) for c in (cam0, cam1)]
tables = decoder.tables(frames)
cameras = {'reset': None, 'table1': decoder.camera_table([cam0], np.zeros(frames, np.int64)),
           'table2': decoder.camera_table([cam0, cam1], np.arange(frames) % 2)}
parts = [(split[0], slice(0, half)), (split[1], slice(half, frames))]


def step(arm, phase):
    """One batch of the arm: phase 'k1', 'group' or 'decode'."""
    calls = [(d, s, None) for d, s in parts] if arm == 'split' else [(decoder, slice(0, frames), cameras[arm])]
    for d, s, table in calls:
        t = d.tables(s.stop - s.start)
        if phase == 'k1':
            d.extract_peaks(heat[s], t)
        elif phase == 'group':
            d.group_objects(depth[s], centers[s], t, cameras=table)
        else:
            d.decode_batch(heat[s], depth[s], centers[s], tables=t, cameras=table)


def timed(arm, phase):
    """us per batch over reps; K1 and grouping each bracketed by events, the peak tables refreshed before a grouping."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    total = 0.0
    if phase == 'decode':
        ev[0].record()
        for _ in range(reps):
            step(arm, 'decode')
        ev[1].record()
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1]) / reps * 1e3
    for _ in range(reps):
        if phase == 'group':
            step(arm, 'k1')
        ev[0].record()
        step(arm, phase)
        ev[1].record()
        torch.cuda.synchronize()
        total += ev[0].elapsed_time(ev[1])
    return total / reps * 1e3


arms = ['reset', 'table1', 'table2', 'split']
for arm in arms:                                              # warm-up: every kernel and shape of every arm
    for phase in ('k1', 'group', 'decode'):
        step(arm, phase)
torch.cuda.synchronize()
results = {arm: {'k1': [], 'group': [], 'decode': []} for arm in arms}
for r in range(rounds):
    for arm in (arms if r % 2 == 0 else arms[::-1]):
        for phase in ('k1', 'group', 'decode'):
            results[arm][phase].append(timed(arm, phase))
# the table arms decode what reset / split decode: one camera per frame either way
reference = decoder.decode_batch(heat, depth, centers, tables=tables).numpy()
same_table1 = all(np.array_equal(v, reference[k]) for k, v in
                  decoder.decode_batch(heat, depth, centers, cameras=cameras['table1']).numpy().items())
summary = {
    'workload': f"{frames} frames of {shape}, keypoint_config {cfg}" + (", lean_tables" if lean else ""),
    'device': torch.cuda.get_device_name(0), 'reps': reps, 'rounds': rounds,
    'us_median': {arm: {phase: float(np.median(v)) for phase, v in ph.items()} for arm, ph in results.items()},
    'us_all': results, 'table1_equals_reset': same_table1,
}
print(json.dumps(summary))
for arm in arms:
    m = summary['us_median'][arm]
    print(f"# {shape} {arm:6s} K1 {m['k1']:8.1f} us  group {m['group']:7.1f} us  decode {m['decode']:8.1f} us")
