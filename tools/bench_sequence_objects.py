"""BASELINE config 3 on the GPU: the 900-frame moving-camera sequence (synthetic_sequence, 180x320, 8 valves, keypoint_config
[1, 3]) at V = 16 views per anchor. Timed with CUDA events as medians of alternating rounds: the decode, the per-peak
chain (SequenceTriangulator.__call__), the sequence-objects C entry in both association modes (okp_triangulate_sequence_
objects_f64 with prepared arguments and preallocated outputs: the matching kernel and the track kernel) and the Python
call (SequenceTriangulator.objects) in both modes. Accuracy lines, for exact depth maps and for depth maps scaled per
frame by up to +-10 %: wrong object matches against the construction (each object identified by the nearest projected
centre), tracks triangulated, median and largest error against the scene in mm, views dropped by the reprojection filter.

    python tools/bench_sequence_objects.py [rounds]

The keypoints carry 0.3 px of Gaussian noise; the maps are rasterised with center_radius 8 so that lifts read at the
undistorted pixel land on their disc (tests/test_gpu_sequence_objects.py does the same).
"""
import ctypes
import os
import statistics
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from object_keypoints_b200 import KeypointDecoder, _lib, sequence, synthetic, targets  # noqa: E402

CFG = [1, 3]
SIZE = (180, 320)
VIEWS = 16


def timed(fn, reps):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        fn()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) / reps


def entry(chain, tables, prepared, out, association):
    """The C entry with every argument prepared once and preallocated outputs: the two launches alone."""
    cfg = (ctypes.c_int32 * len(CFG))(*CFG)
    args = (ctypes.byref(tables.struct), tables.N, tables.C, cfg, ctypes.byref(tables.params), prepared['frames_i32'].data_ptr(),
            out.A, out.V, prepared['F'].data_ptr(), prepared['motion'].data_ptr(), prepared['poses'].data_ptr(),
            ctypes.byref(chain._cam), sequence.SEQUENCE_ASSOCIATIONS.index(association), chain.max_distance_px,
            sequence.DEFAULT_SEQUENCE_MAX_DEPTH_PX, chain.max_error_px, chain.max_rounds, ctypes.byref(out.struct), None)
    function = _lib.lib().okp_triangulate_sequence_objects_f64

    def call():
        _lib.check(function(*args), 'okp_triangulate_sequence_objects_f64')
    call.keep = cfg
    return call


def wrong_matches(t, got, keypoints, frames):
    """(wrong object matches, object matches, largest cost of a right match)"""
    def scene_object(f, o):
        return int(np.linalg.norm(keypoints[f, :, 0] - t['kp_xy'][f, o, 0, 0], axis=1).argmin())
    wrong = total = 0
    right_cost = 0.0
    for a, v, o in zip(*np.nonzero(got['object_match'] >= 0)):
        total += 1
        bad = scene_object(frames[a, 0], o) != scene_object(frames[a, v + 1], got['object_match'][a, v, o])
        wrong += bad
        if not bad:
            right_cost = max(right_cost, float(got['object_cost'][a, v, o]))
    return wrong, total, right_cost


def errors_mm(points, scene):
    ok = ~np.isnan(points[..., 0])
    e = np.linalg.norm(points[ok][:, None] - scene.reshape(-1, 3)[None], axis=2).min(axis=1) * 1e3
    return int(ok.sum()), float(np.median(e)), float(e.max())


def main():
    rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    props = torch.cuda.get_device_properties(0)
    print(f"GPU: {props.name}, {props.multi_processor_count} SMs; power limit: see nvidia-smi lines")
    camera = synthetic.default_camera(SIZE)
    seq = sequence.synthetic_sequence(900)
    keypoints, depths = sequence.project_sequence(seq, camera)
    rng = np.random.default_rng(3)
    noisy = keypoints + rng.normal(0.0, 0.3, keypoints.shape)
    factors = 1.0 + rng.uniform(-0.1, 0.1, 900)
    heat, depth, centers = targets.rasterise_targets(noisy, depths, CFG, SIZE, center_radius=8.0)
    scaled = depth * torch.from_numpy(factors.astype(np.float32)).cuda()[:, None, None, None]
    decoder = KeypointDecoder(CFG, SIZE, camera=camera, compat_clip_bug=False)
    chain = sequence.SequenceTriangulator(camera, views=VIEWS)
    prepared = chain.prepare(seq['T_CW'])
    frames = sequence.view_schedule(900, VIEWS)
    tables = decoder.decode_batch(heat, depth, centers)
    outs = {m: chain.objects(tables, prepared, association=m) for m in sequence.SEQUENCE_ASSOCIATIONS}
    launches = {m: entry(chain, tables, prepared, outs[m], m) for m in outs}
    torch.cuda.synchronize()
    arms = {
        'decode': lambda: decoder.decode_batch(heat, depth, centers, tables=tables),
        'per-peak chain': lambda: chain(tables, prepared),
        'objects entry, epipolar': launches['epipolar'],
        'objects entry, depth': launches['depth'],
        'objects call, epipolar': lambda: chain.objects(tables, prepared),
        'objects call, depth': lambda: chain.objects(tables, prepared, association='depth'),
    }
    for fn in arms.values():                                          # warm-up of every shape
        fn()
    torch.cuda.synchronize()
    timings = {k: [] for k in arms}
    for _ in range(rounds):
        for name, fn in arms.items():
            timings[name].append(timed(fn, 10))
    A = frames.shape[0]
    print(f"900 frames of {SIZE[0]}x{SIZE[1]}, keypoint_config {CFG}, {A} anchors x {VIEWS} views "
          f"({A * (VIEWS - 1)} anchor/view pairs), {int(tables['n_objects'].sum())} decoded objects")
    for name, v in timings.items():
        print(f"  {name:26s} {statistics.median(v):8.3f} ms median of {rounds} rounds x 10 calls (min {min(v):.3f}, max {max(v):.3f})")
    med = {k: statistics.median(v) for k, v in timings.items()}
    print(f"  objects entry / per-peak chain: epipolar {med['objects entry, epipolar'] / med['per-peak chain']:.3f}, "
          f"depth {med['objects entry, depth'] / med['per-peak chain']:.3f}")
    for label, maps in (('exact depth', depth), ('depth maps scaled per frame by up to +-10 %', scaled)):
        t_dev = decoder.decode_batch(heat, maps, centers)
        t = t_dev.numpy()
        peaks = {k: v.cpu().numpy() for k, v in chain(t_dev, prepared).items()}
        n, median, worst = errors_mm(peaks['points'], seq['scene'])
        print(f"accuracy, {label}: per-peak chain: {n} tracks triangulated, error median {median:.2f} mm, max {worst:.1f} mm, "
              f"{int(peaks['dropped'].sum())} views dropped")
        # the depth mode also with a loose gate (64 px): the cost of every right match, where the default gate would cut
        for m, gate in (('epipolar', None), ('depth', sequence.DEFAULT_SEQUENCE_MAX_DEPTH_PX), ('depth', 64.0)):
            kwargs = {} if gate is None else {'max_depth_px': gate}
            got = chain.objects(t_dev, prepared, association=m, **kwargs).numpy()
            wrong, total, right_cost = wrong_matches(t, got, keypoints, frames)
            n, median, worst = errors_mm(got['point'], seq['scene'])
            name = m if gate is None else f"{m} (max_depth_px {gate:g})"
            print(f"accuracy, {label}: objects {name}: {wrong} wrong object matches of {total}, {n} tracks triangulated, "
                  f"error median {median:.2f} mm, max {worst:.1f} mm, {int(got['dropped'].sum())} views dropped, "
                  f"largest cost of a right object match {right_cost:.2f} px, "
                  f"flags {np.bincount(got['flags'].ravel(), minlength=8)[:8].tolist()}")


if __name__ == '__main__':
    main()
