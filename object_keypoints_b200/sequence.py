"""BASELINE config 3: a sequence filmed by a moving camera -> tracks -> robust multi-view triangulation.

The reference triangulates a labelled keypoint from TWO frames of a sequence whose camera poses are known
(``LabelingApp._triangulate``, scripts/label.py:285-305: ``T_RL = inv(T_WR) @ T_WL``, ``P1 = K [I|0]``,
``P2 = K [I|0] T_RL``, undistort, ``cv2.triangulatePoints``; the frame pair is the one farthest apart,
``_find_furthest`` :113-134). north_star generalises that to V views per point with a reprojection-error filter.
This module is the chain for a whole decoded sequence, everything on the device:

    decode tables of N frames (okp_decode_*)                                  peak lists per frame and map
      -> okp_fisheye_undistort_f64                                            pinhole pixels of every peak
      -> okp_associate_pairs_f64                                              each anchor frame against its V - 1 view frames,
                                                                              per map, by epipolar distance under the pair's F
      -> tracks [A, C*K, V]                                                   observation of anchor peak k in every view
      -> okp_triangulate_tracks_f64                                           V-view DLT + reprojection filter + re-solve

``SequenceTriangulator.objects`` is the same chain on the decode tables' objects instead of raw peaks: each anchor frame's
objects are matched into its view frames (by epipolar distance, or by where each frame's depth lift lands in the other
frame), slot by slot, and every anchor keypoint becomes a track of V views, all in one matching kernel
(okp_triangulate_sequence_objects_f64) followed by the same robust track kernel. Its result says which object and slot
each world point belongs to.

Frames are taken in ``views`` strides: anchor a in [0, N // views) is seen again in frames a + v * (N // views).
The synthetic sequence (``synthetic_sequence``) follows SURVEY.md section 8d #3: 900 frames of 180x320, 8 valves on a
4 x 2 grid, camera on a spherical cap r in [0.6, 1.0] m looking at the workspace.
"""
import ctypes

import numpy as np
import torch

from . import _abi, _lib, camera_utils, linalg
from .pipeline import SequenceObjectTables, _device, _stream_handle


def synthetic_sequence(n_frames=900, keypoint_config=(1, 3), grid=(4, 2), spacing=0.22, seed=1003):
    """-> dict(scene [G,Kp,3] world points with each object's centre (mean of its keypoints, video.py:128) first,
    T_CW [N,4,4] world->camera, T_WC [N,4,4])."""
    rng = np.random.default_rng(seed)
    gx, gy = grid
    Kp = 1 + int(sum(keypoint_config))
    scene = np.zeros((gx * gy, Kp, 3))
    for o in range(gx * gy):
        base = np.array([(o % gx - (gx - 1) / 2) * spacing, (o // gx - (gy - 1) / 2) * spacing, 0.0])
        base[:2] += rng.uniform(-0.02, 0.02, 2)
        points = []
        for count in keypoint_config:
            if count == 1:                                   # the valve's knob: above the plane
                points.append(base + np.array([0.0, 0.0, -0.05]) + rng.uniform(-0.005, 0.005, 3))
            else:                                            # spokes in the plane
                phase = rng.uniform(0, 2 * np.pi)
                for k in range(count):
                    angle = phase + 2 * np.pi * k / count + rng.uniform(-0.15, 0.15)
                    points.append(base + 0.05 * np.array([np.cos(angle), np.sin(angle), 0.0]))
        points = np.array(points)
        scene[o, 0] = points.mean(axis=0)
        scene[o, 1:] = points
    t = np.linspace(0.0, 1.0, n_frames)
    azimuth = 2 * np.pi * 2.5 * t
    polar = np.deg2rad(8.0 + 14.0 * (0.5 + 0.5 * np.sin(2 * np.pi * 1.7 * t)))
    radius = 0.8 + 0.2 * np.sin(2 * np.pi * 1.1 * t + 0.3)
    T_WC = np.tile(np.eye(4), (n_frames, 1, 1))
    for n in range(n_frames):
        # the camera looks along +z at the workspace, which lies "below" it in world -z ... world z points away from the camera
        position = radius[n] * np.array([np.sin(polar[n]) * np.cos(azimuth[n]), np.sin(polar[n]) * np.sin(azimuth[n]),
                                         -np.cos(polar[n])])
        target = np.array([0.03 * np.sin(7 * t[n]), 0.02 * np.cos(5 * t[n]), 0.0])
        z = target - position
        z /= np.linalg.norm(z)
        x = np.cross(np.array([0.0, 1.0, 0.0]), z)
        x /= np.linalg.norm(x)
        y = np.cross(z, x)
        T_WC[n, :3, 0], T_WC[n, :3, 1], T_WC[n, :3, 2], T_WC[n, :3, 3] = x, y, z, position
    T_CW = np.stack([linalg.inv_transform(T) for T in T_WC])
    return {'scene': scene, 'T_CW': T_CW, 'T_WC': T_WC}


def project_sequence(sequence, camera):
    """Projects the scene into every frame: -> keypoints [N,G,Kp,2] (x, y) pixels, depths [N,G,Kp] camera-frame z --
    the inputs of targets.rasterise_targets (what perception/datasets/video.py:117-129 computes per frame)."""
    scene, T_CW = sequence['scene'], sequence['T_CW']
    G, Kp = scene.shape[:2]
    N = T_CW.shape[0]
    keypoints = np.zeros((N, G, Kp, 2))
    depths = np.zeros((N, G, Kp))
    flat = scene.reshape(-1, 3)
    for n in range(N):
        keypoints[n] = camera.project(flat, T_CW[n]).reshape(G, Kp, 2)
        depths[n] = (flat @ T_CW[n, :3, :3].T + T_CW[n, :3, 3])[:, 2].reshape(G, Kp)
    return keypoints, depths


def view_schedule(n_frames, views):
    """-> frames [A, V]: anchor a = frames[a, 0] is seen again in frames[a, 1:], ``n_frames // views`` frames apart."""
    stride = n_frames // views
    if stride < 1:
        raise ValueError("fewer frames than views")
    return np.arange(stride)[:, None] + stride * np.arange(views)[None, :]


def pair_fundamentals(camera, T_CW, frames):
    """F [A, V-1, 3, 3] with x_view^T F x_anchor = 0 for undistorted pixels: the pair geometry of scripts/label.py:285-297
    (T_RL = T_CW[view] @ inv(T_CW[anchor])) turned into camera_utils.fundamental_matrix (camera_utils.py:184-189)."""
    A, V = frames.shape
    K = np.asarray(camera.K, dtype=np.float64)
    F = np.zeros((A, V - 1, 3, 3))
    for a in range(A):
        T_anchor_inv = linalg.inv_transform(T_CW[frames[a, 0]])
        for v in range(1, V):
            F[a, v - 1] = camera_utils.fundamental_matrix(T_CW[frames[a, v]] @ T_anchor_inv, K, K)
    return F


def pair_motions(T_CW, frames):
    """motion [A, V-1, 2, 12]: for each (anchor, view) pair the rigid motion T = T_CW[view] inv(T_CW[anchor]) (anchor camera ->
    view camera; the T_RL of pair_fundamentals) as (R row-major, t), then its inverse as (R^T, -R^T t), the inverse formed
    in the operation order okp_triangulate_stereo_objects_depth_f64 uses for T_RL."""
    A, V = frames.shape
    motion = np.zeros((A, V - 1, 2, 12))
    for a in range(A):
        T_anchor_inv = linalg.inv_transform(T_CW[frames[a, 0]])
        for v in range(1, V):
            T = T_CW[frames[a, v]] @ T_anchor_inv
            R, t = T[:3, :3], T[:3, 3]
            motion[a, v - 1, 0, :9], motion[a, v - 1, 0, 9:] = R.reshape(9), t
            motion[a, v - 1, 1, :9] = R.T.reshape(9)
            motion[a, v - 1, 1, 9:] = [-(R[0, r] * t[0] + R[1, r] * t[1] + R[2, r] * t[2]) for r in range(3)]
    return motion


SEQUENCE_ASSOCIATIONS = ('epipolar', 'depth')
# DESIGN.md section 3 (sequence objects): the worst true-pair depth cost of this sequence's pairs at a +-10 % depth error
DEFAULT_SEQUENCE_MAX_DEPTH_PX = 16.0


def anchor_objects(result, a):
    """One anchor's objects from the host copy (``SequenceObjectTables.numpy()``) of SequenceTriangulator.objects, in the
    structure tables_to_objects gives a frame: a list (one entry per anchor object) of dicts with 'keypoints' (per map, the
    anchor's distorted pixels [k, 2], an empty array where the object has none) and 'p_W' (per map, the world points
    [k, 3], NaN where a track had fewer than two valid views; None where the object has no keypoint of that map)."""
    observed = result['observed'][a, ..., 0].astype(bool)                  # [O, C, S]: the anchor's own keypoints
    objects = []
    for o in range(observed.shape[0]):
        if not observed[o, 0, 0]:
            continue
        keypoints, points = [], []
        for c in range(observed.shape[1]):
            k = int(observed[o, c].sum())
            keypoints.append(result['observations'][a, o, c, :k, 0].copy() if k else np.array([]))
            points.append(result['point'][a, o, c, :k].copy() if k else None)
        objects.append({'keypoints': keypoints, 'p_W': points})
    return objects


class SequenceTriangulator:
    """decode tables of a sequence + its camera poses -> one 3D point per anchor peak (world frame)."""

    def __init__(self, camera, views=16, max_distance_px=2.5, max_error_px=2.0, max_rounds=None, device=None):
        self.camera = camera
        self.views = int(views)
        self.max_distance_px = float(max_distance_px)
        self.max_error_px = float(max_error_px)
        self.max_rounds = self.views if max_rounds is None else int(max_rounds)
        self.device = _device(device)
        self._cam = _abi.pack_camera(camera)
        self._lib = _lib.lib()

    def prepare(self, T_CW):
        """Host-side, once per sequence: the view schedule, the poses of every track group and the pair geometry
        (F for both calls; for ``objects`` also the schedule as int32, the pairs' rigid motions and the frame count)."""
        T_CW = np.asarray(T_CW, dtype=np.float64)
        frames = view_schedule(T_CW.shape[0], self.views)
        F = pair_fundamentals(self.camera, T_CW, frames)
        return {'frames': torch.from_numpy(frames).to(self.device),
                'poses': torch.from_numpy(np.ascontiguousarray(T_CW[frames])).to(self.device),           # [A, V, 4, 4]
                'F': torch.from_numpy(F).to(self.device),
                'frames_i32': torch.from_numpy(frames.astype(np.int32)).to(self.device),
                'motion': torch.from_numpy(pair_motions(T_CW, frames)).to(self.device),                   # [A, V-1, 2, 12]
                'n_frames': int(T_CW.shape[0])}

    def __call__(self, tables, prepared, stream=None):
        """tables: DecodeTables (or a dict of CUDA tensors) of the N frames. -> dict of CUDA tensors:
        points [A, C, K, 3] world frame (NaN where a track has fewer than two views), valid [A, C, K, V] uint8 after the
        reprojection filter, error [A, C, K, V] px, dropped [A, C, K], observed [A, C, K, V] uint8 before the filter,
        match [A, V-1, C, K] index of the anchor peak's partner in the view frame or -1."""
        t = tables.tensors if hasattr(tables, 'tensors') else tables
        lib, handle = self._lib, _stream_handle(stream)
        N, C, K = (int(v) for v in t['peak_xy'].shape[:3])
        frames, poses, F = prepared['frames'], prepared['poses'], prepared['F']
        A, V = (int(v) for v in frames.shape)
        xy = t['peak_xy'].to(torch.float64).contiguous()                                  # [N, C, K, 2] distorted pixels
        undistorted = torch.empty_like(xy)
        rc = lib.okp_fisheye_undistort_f64(xy.data_ptr(), N * C * K, ctypes.byref(self._cam), 0, undistorted.data_ptr(), handle)
        _lib.check(rc, 'okp_fisheye_undistort_f64')
        count = t['peak_count'].clamp(max=K).to(torch.int32)                              # [N, C]
        anchor, others = frames[:, 0], frames[:, 1:]                                      # [A], [A, V-1]
        B = A * (V - 1) * C
        left = undistorted[anchor][:, None].expand(A, V - 1, C, K, 2).contiguous()        # pair (a, v, c): anchor's map c
        right = undistorted[others].contiguous()                                          # [A, V-1, C, K, 2]
        n_left = count[anchor][:, None].expand(A, V - 1, C).contiguous()
        n_right = count[others].contiguous()
        F_pairs = F[:, :, None].expand(A, V - 1, C, 3, 3).contiguous()
        match = torch.empty((A, V - 1, C, K), dtype=torch.int32, device=self.device)
        cost = torch.empty((A, V - 1, C, K), dtype=torch.float64, device=self.device)
        rc = lib.okp_associate_pairs_f64(F_pairs.data_ptr(), left.data_ptr(), n_left.data_ptr(), right.data_ptr(),
                                         n_right.data_ptr(), B, K, K, self.max_distance_px, match.data_ptr(), cost.data_ptr(), handle)
        _lib.check(rc, 'okp_associate_pairs_f64')
        # tracks: the anchor's own (distorted) observation, then its partner's in every view
        obs = torch.zeros((A, C, K, V, 2), dtype=torch.float64, device=self.device)
        observed = torch.zeros((A, C, K, V), dtype=torch.uint8, device=self.device)
        real = torch.arange(K, device=self.device)[None, None, :] < count[anchor][:, :, None]          # [A, C, K]
        obs[:, :, :, 0] = xy[anchor]
        observed[:, :, :, 0] = real.to(torch.uint8)
        m = match.permute(0, 2, 3, 1)                                                                    # [A, C, K, V-1]
        partner = xy[others].permute(0, 2, 1, 3, 4)                                                      # [A, C, V-1, K, 2]
        index = m.clamp(min=0).permute(0, 1, 3, 2)[..., None].expand(A, C, V - 1, K, 2).to(torch.int64)
        picked = torch.gather(partner, 3, index).permute(0, 1, 3, 2, 4)                                  # [A, C, K, V-1, 2]
        seen = (m >= 0) & real[..., None]
        obs[:, :, :, 1:] = torch.where(seen[..., None], picked, torch.zeros((), dtype=torch.float64, device=self.device))
        observed[:, :, :, 1:] = seen.to(torch.uint8)
        valid = observed.clone()
        points = torch.empty((A, C, K, 3), dtype=torch.float64, device=self.device)
        error = torch.empty((A, C, K, V), dtype=torch.float64, device=self.device)
        dropped = torch.zeros((A, C, K), dtype=torch.int32, device=self.device)
        rc = lib.okp_triangulate_tracks_f64(obs.data_ptr(), valid.data_ptr(), poses.data_ptr(), ctypes.byref(self._cam), A, C * K, V,
                                            self.max_error_px, self.max_rounds, points.data_ptr(), error.data_ptr(),
                                            dropped.data_ptr(), handle)
        _lib.check(rc, 'okp_triangulate_tracks_f64')
        return {'points': points, 'valid': valid, 'error': error, 'dropped': dropped, 'observed': observed, 'match': match,
                'observations': obs}

    def objects(self, tables, prepared, association='epipolar', max_depth_px=DEFAULT_SEQUENCE_MAX_DEPTH_PX, stream=None):
        """The decoded objects of the sequence, per anchor and slot, triangulated in the world frame
        (okp_triangulate_sequence_objects_f64). tables: the DecodeTables of the N frames ``prepare`` was given, decoded with
        this camera. Each anchor frame's objects are matched into its V - 1 view frames by their centres, then each matched
        object's slots type by type, greedily one to one: association='epipolar' by the epipolar distance under the pair's
        F while it is <= max_distance_px (triangulate_stereo_objects' rule); association='depth' by where each keypoint's
        lift (kp_point) lands in the other frame, over the candidates within max_distance_px of the epipolar line and with
        d <= max_depth_px (the stereo depth rule), which tells apart objects that lie on one epipolar line of a view. The
        matches of every anchor slot form a track of V views, solved like ``__call__`` solves peak tracks (V-view DLT,
        reprojection filter with max_error_px, re-solve). ValueError for an unknown mode, tables of another frame count
        than the prepared poses, and association='depth' on tables decoded with compat_clip_bug when the camera's image is
        not square (such lifts read the depth of a clipped column). Returns SequenceObjectTables on the tables' device;
        asynchronous: nothing synchronises. anchor_objects(result.numpy(), a) gives anchor a's objects as dicts."""
        if association not in SEQUENCE_ASSOCIATIONS:
            raise ValueError(f"association must be one of {SEQUENCE_ASSOCIATIONS}, got {association!r}")
        if tables.N != prepared['n_frames']:
            raise ValueError(f"the tables hold {tables.N} frames, the prepared poses {prepared['n_frames']}")
        if association == 'depth':
            size = np.asarray(self.camera.image_size).reshape(-1)[:2]
            if tables.params.compat_clip_bug and size[0] != size[1]:
                raise ValueError("association='depth' reads kp_point, and with compat_clip_bug a non-square image is lifted "
                                 "with the depth of a clipped column: decode with compat_clip_bug=False")
        frames = prepared['frames_i32']
        A, V = (int(v) for v in frames.shape)
        O, C, S = (int(v) for v in tables['kp_xy'].shape[1:4])
        device = tables.flat.device
        out = SequenceObjectTables(A, V, O, C, S, device)
        cfg = (ctypes.c_int32 * max(len(tables.keypoint_config), 1))(*tables.keypoint_config)
        with torch.cuda.device(device):
            rc = self._lib.okp_triangulate_sequence_objects_f64(
                ctypes.byref(tables.struct), tables.N, C, cfg, ctypes.byref(tables.params), frames.data_ptr(), A, V,
                prepared['F'].data_ptr(), prepared['motion'].data_ptr(), prepared['poses'].data_ptr(), ctypes.byref(self._cam),
                SEQUENCE_ASSOCIATIONS.index(association), self.max_distance_px, float(max_depth_px), self.max_error_px,
                self.max_rounds, ctypes.byref(out.struct), _stream_handle(stream))
        _lib.check(rc, 'okp_triangulate_sequence_objects_f64')
        out.prepared = prepared                              # the launch reads its arrays: kept alive with the result
        return out
