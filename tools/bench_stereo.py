"""Stereo objects on the GPU: the decode call and the triangulate_stereo_objects call on the same stereo batch, timed with
CUDA events as medians of alternating rounds, plus the C entry alone (preallocated outputs: the kernel without the Python
wrapper's per-call work), the grouping kernel alone on the same frames and the host-level loop
(AssociationComponent + TriangulationComponent per pair and keypoint type) on a subset of the pairs. Both association
modes are timed in the same rounds, 'epipolar' and 'depth' (whose lifts need compat_clip_bug off at 180x320: the decoder
runs without it for both). An accuracy line per size counts the wrong matches of each mode on a batch of same-row pairs
(two objects per pair, centre rows within 0.3 px: side by side on one epipolar line).

    python tools/bench_stereo.py [rounds]

Batches: config 2 (64 pairs of 64x64 cups frames [1,1,1], 1-4 objects) and a large one (2048 pairs of 180x320 valve
frames [1,3], 1-4 objects; 32 distinct pairs generated on the host, repeated 64 times on the device -- the maps are 9 GB,
far beyond L2, so repetition does not make the decode cheaper).
"""
import os
import statistics
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from object_keypoints_b200 import (AssociationComponent, KeypointDecoder, TriangulationComponent,  # noqa: E402
                                   synthetic, triangulate_stereo_objects)


def timed(fn, reps):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        fn()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) / reps


def host_loop(tables, stereo, pairs, cfg):
    """The per-point host components on the decoded tables: one association of the centres per pair, then one association
    and one triangulation per matched object and keypoint type (every call copies through the host)."""
    association, triangulation = AssociationComponent(), TriangulationComponent()
    association.reset(stereo)
    triangulation.reset(stereo)
    t = {k: tables[k].cpu().numpy() for k in ('n_objects', 'kp_count', 'kp_xy')}
    began = time.perf_counter()
    for l, r in pairs:
        nl, nr = int(t['n_objects'][l]), int(t['n_objects'][r])
        match = association(t['kp_xy'][l, :nl, 0, 0], t['kp_xy'][r, :nr, 0, 0])
        for i, j in enumerate(match.tolist()):
            if j < 0:
                continue
            for c in range(len(cfg) + 1):
                left = t['kp_xy'][l, i, c, :t['kp_count'][l, i, c]]
                right = t['kp_xy'][r, j, c, :t['kp_count'][r, j, c]]
                slots = association(left, right) if c else np.zeros(1, np.int64)
                keep = slots >= 0
                if keep.any():
                    triangulation(left[keep], right[slots[keep]])
    return (time.perf_counter() - began) * 1e3


def entry(tables, stereo, out, optimal_correction=True, association='epipolar'):
    """The C entry with every argument prepared once and preallocated outputs: the launch alone, without the Python
    wrapper's per-call work (camera packing, output allocation, the default pair table)."""
    import ctypes
    from object_keypoints_b200 import _abi, _lib
    keep = [(ctypes.c_int32 * len(tables.keypoint_config))(*tables.keypoint_config),
            _abi.pack_camera(stereo.left_camera), _abi.pack_camera(stereo.right_camera)]
    matrices = [np.ascontiguousarray(m, dtype=np.float64) for m in (stereo.F, *stereo.projection_matrices())]
    doubles = ctypes.POINTER(ctypes.c_double)
    head = (ctypes.byref(tables.struct), tables.N, tables.C, keep[0], ctypes.byref(tables.params), out.pairs.data_ptr(),
            out.P, ctypes.byref(keep[1]), ctypes.byref(keep[2]), *(m.ctypes.data_as(doubles) for m in matrices))
    lib = _lib.lib()
    if association == 'depth':
        matrices.append(np.ascontiguousarray(stereo.T_RL, dtype=np.float64).reshape(16))
        args = (*head, matrices[-1].ctypes.data_as(doubles), 2.5, 8.0, int(optimal_correction), ctypes.byref(out.struct), None)
        name = 'okp_triangulate_stereo_objects_depth_f64'
    else:
        args = (*head, 2.5, int(optimal_correction), ctypes.byref(out.struct), None)
        name = 'okp_triangulate_stereo_objects_f64'
    function = getattr(lib, name)

    def call():
        _lib.check(function(*args), name)
    call.keep = (keep, matrices)
    return call


def run(name, size, cfg, pairs, distinct, rounds, reps, host_pairs):
    stereo = synthetic.stereo_rig(size)
    sb = synthetic.stereo_batch(distinct, cfg, size, stereo, seed=21)
    maps = [torch.from_numpy(a).cuda().repeat((pairs // distinct,) + (1,) * (a.ndim - 1))
            for a in (sb.batch.heat, sb.batch.depth, sb.batch.centers)]
    N = maps[0].shape[0]
    decoder = KeypointDecoder(cfg, size, compat_clip_bug=False)
    cameras = decoder.camera_table((stereo.left_camera, stereo.right_camera), np.arange(N) % 2)
    tables = decoder.decode_batch(*maps, cameras=cameras)
    out = triangulate_stereo_objects(tables, stereo)
    out_depth = triangulate_stereo_objects(tables, stereo, association='depth')
    torch.cuda.synchronize()
    timings = {'decode': [], 'grouping': [], 'stereo': [], 'stereo, no correction': [], 'stereo kernel': [],
               'stereo kernel, no corr.': [], 'depth': [], 'depth, no correction': [], 'depth kernel': [],
               'depth kernel, no corr.': []}
    launch, launch_plain = entry(tables, stereo, out), entry(tables, stereo, out, optimal_correction=False)
    launch_depth = entry(tables, stereo, out_depth, association='depth')
    launch_depth_plain = entry(tables, stereo, out_depth, optimal_correction=False, association='depth')
    for _ in range(rounds):
        timings['decode'].append(timed(lambda: decoder.decode_batch(*maps, tables=tables, cameras=cameras), reps))
        timings['grouping'].append(timed(lambda: decoder.group_objects(maps[1], maps[2], tables, cameras=cameras), reps))
        timings['stereo'].append(timed(lambda: triangulate_stereo_objects(tables, stereo), reps))
        timings['stereo, no correction'].append(
            timed(lambda: triangulate_stereo_objects(tables, stereo, optimal_correction=False), reps))
        timings['stereo kernel'].append(timed(launch, reps))
        timings['stereo kernel, no corr.'].append(timed(launch_plain, reps))
        timings['depth'].append(timed(lambda: triangulate_stereo_objects(tables, stereo, association='depth'), reps))
        timings['depth, no correction'].append(
            timed(lambda: triangulate_stereo_objects(tables, stereo, optimal_correction=False, association='depth'), reps))
        timings['depth kernel'].append(timed(launch_depth, reps))
        timings['depth kernel, no corr.'].append(timed(launch_depth_plain, reps))
    launch()
    launch_depth()
    got = out.numpy()
    got_depth = out_depth.numpy()
    matched = int((got['slot_match'] >= 0).sum())
    host_ms = host_loop(tables, stereo, [(2 * p, 2 * p + 1) for p in range(host_pairs)], cfg)
    med = {k: statistics.median(v) for k, v in timings.items()}
    spread = {k: (min(v), max(v)) for k, v in timings.items()}
    print(f"{name}: {pairs} pairs ({N} frames) of {size[0]}x{size[1]}, keypoint_config {cfg}, "
          f"{int(tables['n_objects'].sum())} objects, {int((got['object_match'] >= 0).sum())} object matches, "
          f"{matched} keypoint pairs triangulated, flags set on {int((got['flags'] != 0).sum())} pairs; depth mode: "
          f"{int((got_depth['object_match'] >= 0).sum())} object matches, {int((got_depth['slot_match'] >= 0).sum())} keypoint "
          f"pairs, flags set on {int((got_depth['flags'] != 0).sum())} pairs")
    for k in timings:
        print(f"  {k:22s} {med[k]:8.3f} ms median of {rounds} rounds x {reps} calls (min {spread[k][0]:.3f}, max {spread[k][1]:.3f})")
    print(f"  stereo call / decode call {med['stereo'] / med['decode']:.3f}; stereo kernel / grouping "
          f"{med['stereo kernel'] / med['grouping']:.3f}; stereo kernel per pair {1e3 * med['stereo kernel'] / pairs:.3f} us; "
          f"depth kernel / stereo kernel {med['depth kernel'] / med['stereo kernel']:.3f}")
    print(f"  host loop (AssociationComponent + TriangulationComponent per pair and type): {host_ms:.1f} ms for {host_pairs} "
          f"pairs = {host_ms / host_pairs:.2f} ms per pair, {host_ms / host_pairs * pairs:.0f} ms for the batch (extrapolated)")


def accuracy(size, cfg, pairs):
    """Wrong matches of each association mode on same-row pairs, against the construction (synthetic.stereo_match_errors)."""
    stereo = synthetic.stereo_rig(size)
    sb = synthetic.stereo_batch(pairs, cfg, size, stereo, seed=5, objects=(2, 2), same_row=True, row_jitter=0.3,
                                slot_margin=-1.0, max_tries=200000)
    decoder = KeypointDecoder(cfg, size, compat_clip_bug=False)
    cameras = decoder.camera_table((stereo.left_camera, stereo.right_camera), np.arange(2 * pairs) % 2)
    tables = decoder.decode_batch(sb.batch.heat, sb.batch.depth, sb.batch.centers, cameras=cameras)
    t = tables.numpy()
    line = []
    for association in ('epipolar', 'depth'):
        got = triangulate_stereo_objects(tables, stereo, association=association).numpy()
        objects, slots, worst = synthetic.stereo_match_errors(sb, t, got)
        line.append(f"{association}: {objects} wrong object matches, {slots} wrong slot matches, flags set on "
                    f"{int((got['flags'] != 0).sum())} pairs, largest relative point error of a right match {worst:.3g}")
    print(f"same-row accuracy, {pairs} pairs of {size[0]}x{size[1]} {cfg}, {2 * pairs} left objects: " + "; ".join(line))


def main():
    rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    props = torch.cuda.get_device_properties(0)
    print(f"GPU: {props.name}, {props.multi_processor_count} SMs; power limit: see nvidia-smi lines")
    run('config 2', (64, 64), [1, 1, 1], 64, 64, rounds, 50, 16)
    run('large', (180, 320), [1, 3], 2048, 32, rounds, 10, 16)
    accuracy((64, 64), [1, 1, 1], 64)
    accuracy((180, 320), [1, 3], 32)


if __name__ == '__main__':
    main()
