"""Camera geometry and triangulation on the GPU (libokp.so), behind the reference's names.

* ``undistort_points`` / ``project_points`` -- FisheyeCamera.undistort / .project
  (perception/utils/camera_utils.py:65-81) for arrays of points;
* ``triangulate`` -- batched V-view DLT; at V = 2 it is cv2.triangulatePoints as used by
  StereoCamera.triangulate (camera_utils.py:103-108) and LabelingApp._triangulate
  (scripts/label.py:296-305);
* ``TriangulationComponent`` -- the ``reset(stereo)`` / ``__call__(left, right)`` component the
  reference's test-suite expects (test/test_pipeline.py:171-177), pairs matched by index;
* ``triangulate_multiview`` -- undistort, DLT over V views, reprojection-error gate, re-solve;
* ``correct_matches`` -- cv2.correctMatches (Hartley-Sturm) as camera_utils.py:100-101 uses it;
* ``AssociationComponent`` / ``associate`` -- stereo association by epipolar distance
  (test/test_pipeline.py:208-261);
* ``triangulate_stereo_objects`` -- both halves on the decode tables of a stereo batch in one call: objects and
  keypoints matched across the two views, corrected and triangulated in the left camera's frame.
"""
import ctypes

import numpy as np
import torch

from . import _abi, _lib
from .pipeline import StereoTables, _device, _stream_handle


def _as_f64(x, device):
    if isinstance(x, np.ndarray):
        x = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64))
    return x.to(device=device, dtype=torch.float64).contiguous()


def undistort_points(xy, camera, round_to_f32=False, device=None):
    """[n,2] distorted pixels -> [n,2] float64 CUDA tensor of pinhole pixels."""
    device = _device(device)
    xy = _as_f64(xy, device)
    out = torch.empty_like(xy)
    cam = _abi.pack_camera(camera)
    rc = _lib.lib().okp_fisheye_undistort_f64(xy.data_ptr(), xy.shape[0], ctypes.byref(cam), int(round_to_f32),
                                              out.data_ptr(), _stream_handle())
    _lib.check(rc, 'okp_fisheye_undistort_f64')
    return out


def project_points(X, T_CW, camera, device=None):
    """[n,3] points, 4x4 world->camera -> [n,2] float64 CUDA tensor of distorted pixels."""
    device = _device(device)
    X = _as_f64(X, device)
    out = torch.empty((X.shape[0], 2), dtype=torch.float64, device=device)
    cam = _abi.pack_camera(camera)
    T = np.ascontiguousarray(np.asarray(T_CW, dtype=np.float64).reshape(-1)[:16])
    rc = _lib.lib().okp_fisheye_project_f64(X.data_ptr(), X.shape[0], T.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                            ctypes.byref(cam), out.data_ptr(), _stream_handle())
    _lib.check(rc, 'okp_fisheye_project_f64')
    return out


def triangulate(points, projections, valid=None, device=None):
    """points [P,V,2] undistorted pixels, projections [V,3,4] (shared) or [P,V,3,4], valid [P,V]
    -> [P,3] float64 CUDA tensor (NaN where fewer than two valid views)."""
    device = _device(device)
    points = _as_f64(points, device)
    projections = _as_f64(projections, device)
    P, V = int(points.shape[0]), int(points.shape[1])
    per_point = int(projections.dim() == 4)
    valid_ptr = None
    if valid is not None:
        if isinstance(valid, np.ndarray):
            valid = torch.from_numpy(np.ascontiguousarray(valid))
        valid = valid.to(device=device, dtype=torch.uint8).contiguous()
        valid_ptr = valid.data_ptr()
    out = torch.empty((P, 3), dtype=torch.float64, device=device)
    rc = _lib.lib().okp_triangulate_f64(points.data_ptr(), valid_ptr, projections.data_ptr(), per_point, P, V,
                                        out.data_ptr(), _stream_handle())
    _lib.check(rc, 'okp_triangulate_f64')
    return out


def reprojection_filter(X, observations, valid, poses, camera, max_error_px, device=None):
    """X [P,3], observations [P,V,2] distorted pixels, valid [P,V], poses [V,4,4] world->camera ->
    (valid' [P,V] uint8, error [P,V] float64): views with error > max_error_px are cleared."""
    device = _device(device)
    X = _as_f64(X, device)
    observations = _as_f64(observations, device)
    poses = _as_f64(poses, device)
    P, V = int(observations.shape[0]), int(observations.shape[1])
    if isinstance(valid, np.ndarray):
        valid = torch.from_numpy(np.ascontiguousarray(valid))
    valid = valid.to(device=device, dtype=torch.uint8).contiguous().clone()
    err = torch.empty((P, V), dtype=torch.float64, device=device)
    cam = _abi.pack_camera(camera)
    rc = _lib.lib().okp_reprojection_filter_f64(X.data_ptr(), observations.data_ptr(), valid.data_ptr(), poses.data_ptr(),
                                                ctypes.byref(cam), P, V, float(max_error_px), err.data_ptr(),
                                                _stream_handle())
    _lib.check(rc, 'okp_reprojection_filter_f64')
    return valid, err


def triangulate_multiview(observations, valid, poses, camera, max_error_px=2.0, max_rounds=None, device=None,
                          return_dropped=False):
    """Config-3 path in ONE kernel (okp_triangulate_robust_f64): observations [P,V,2] distorted pixels
    seen from poses [V,4,4] (world->camera) with one equidistant camera. Per point: undistort, V-view
    DLT, reprojection error per view; while the worst valid view is farther than max_error_px (and
    more than two views remain, at most max_rounds drops) drop it and solve again.
    Returns (X [P,3], valid [P,V] uint8, error [P,V]) CUDA tensors."""
    device = _device(device)
    observations = _as_f64(observations, device)
    P, V = int(observations.shape[0]), int(observations.shape[1])
    poses_t = _as_f64(poses, device)
    if valid is None:
        valid = torch.ones((P, V), dtype=torch.uint8, device=device)
    else:
        if isinstance(valid, np.ndarray):
            valid = torch.from_numpy(np.ascontiguousarray(valid))
        valid = valid.to(device=device, dtype=torch.uint8).contiguous().clone()
    X = torch.empty((P, 3), dtype=torch.float64, device=device)
    err = torch.empty((P, V), dtype=torch.float64, device=device)
    dropped = torch.zeros((P,), dtype=torch.int32, device=device)
    cam = _abi.pack_camera(camera)
    rounds = V if max_rounds is None else int(max_rounds)
    rc = _lib.lib().okp_triangulate_robust_f64(observations.data_ptr(), valid.data_ptr(), poses_t.data_ptr(),
                                               ctypes.byref(cam), P, V, float(max_error_px), rounds, X.data_ptr(),
                                               err.data_ptr(), dropped.data_ptr(), _stream_handle())
    _lib.check(rc, 'okp_triangulate_robust_f64')
    if return_dropped:
        return X, valid, err, dropped
    return X, valid, err


def correct_matches(F, left, right, round_to_f32=False, device=None):
    """cv2.correctMatches (camera_utils.py:100-101) on the GPU: [n,2] UNDISTORTED pixel pairs ->
    the closest pairs that satisfy x_right^T F x_left = 0 (Hartley-Sturm). Returns two [n,2] float64
    CUDA tensors."""
    device = _device(device)
    left = _as_f64(left, device)
    right = _as_f64(right, device)
    if left.shape != right.shape or left.dim() != 2 or left.shape[1] != 2:
        raise ValueError(f"correct_matches wants two [n,2] arrays, got {tuple(left.shape)} and {tuple(right.shape)}")
    out_left = torch.empty_like(left)
    out_right = torch.empty_like(right)
    Fm = np.ascontiguousarray(np.asarray(F, dtype=np.float64).reshape(9))
    rc = _lib.lib().okp_correct_matches_f64(Fm.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), left.data_ptr(),
                                            right.data_ptr(), int(left.shape[0]), int(round_to_f32),
                                            out_left.data_ptr(), out_right.data_ptr(), _stream_handle())
    _lib.check(rc, 'okp_correct_matches_f64')
    return out_left, out_right


def associate(F, left, right, n_left=None, n_right=None, max_distance_px=2.5, device=None):
    """Batched stereo association: left [B,ML,2], right [B,MR,2] UNDISTORTED pixels (+ optional valid
    counts [B]) -> (match [B,ML] int32: index into right or -1, cost [B,ML] float64 pixels)."""
    device = _device(device)
    left = _as_f64(left, device)
    right = _as_f64(right, device)
    B, ML, MR = int(left.shape[0]), int(left.shape[1]), int(right.shape[1])

    def counts(n, full):
        if n is None:
            return torch.full((B,), full, dtype=torch.int32, device=device)
        if isinstance(n, np.ndarray):
            n = torch.from_numpy(np.ascontiguousarray(n))
        return torch.as_tensor(n).to(device=device, dtype=torch.int32).contiguous()
    n_left = counts(n_left, ML)
    n_right = counts(n_right, MR)
    match = torch.empty((B, max(ML, 1)), dtype=torch.int32, device=device)
    cost = torch.empty((B, max(ML, 1)), dtype=torch.float64, device=device)
    if ML == 0 or MR == 0:
        return match[:, :ML].fill_(-1), cost[:, :ML].zero_()
    Fm = np.ascontiguousarray(np.asarray(F, dtype=np.float64).reshape(9))
    rc = _lib.lib().okp_stereo_associate_f64(Fm.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), left.data_ptr(),
                                             n_left.data_ptr(), right.data_ptr(), n_right.data_ptr(), B, ML, MR,
                                             float(max_distance_px), match.data_ptr(), cost.data_ptr(),
                                             _stream_handle())
    _lib.check(rc, 'okp_stereo_associate_f64')
    return match, cost


class AssociationComponent:
    """The component test/test_pipeline.py:208-261 expects (its implementation is gone from the
    reference): ``reset(stereo_camera)`` then ``__call__(left[nL,2], right[nR,2])`` distorted pixels ->
    int array [nL], the index of the matching right point or -1. Points are undistorted, then matched
    one-to-one by epipolar distance under ``stereo_camera.F`` (okp_stereo_associate_f64)."""
    name = "association"

    def __init__(self, max_distance_px=2.5):
        self.max_distance_px = max_distance_px
        self.stereo_camera = None

    def reset(self, stereo_camera):
        self.stereo_camera = stereo_camera

    def __call__(self, left_keypoints, right_keypoints):
        left = np.asarray(left_keypoints, dtype=np.float64).reshape(-1, 2)
        right = np.asarray(right_keypoints, dtype=np.float64).reshape(-1, 2)
        if left.shape[0] == 0 or right.shape[0] == 0:
            return np.full((left.shape[0],), -1, dtype=np.int64)
        uL = undistort_points(left, self.stereo_camera.left_camera)
        uR = undistort_points(right, self.stereo_camera.right_camera)
        match, _ = associate(self.stereo_camera.F, uL[None], uR[None], max_distance_px=self.max_distance_px)
        return match[0].cpu().numpy().astype(np.int64)


def triangulate_stereo(stereo, left_keypoints, right_keypoints, optimal_correction=True):
    """StereoCamera.triangulate (camera_utils.py:92-110) on the GPU: float32 cast, undistort both
    views, Hartley-Sturm correction (cv2.correctMatches; ``optimal_correction=False`` gives the plain
    DLT of scripts/label.py:296-305), two-view DLT. Returns [N,3] float64 NumPy in the left camera
    frame."""
    left = np.asarray(left_keypoints).astype(np.float32).astype(np.float64)      # camera_utils.py:93-94
    right = np.asarray(right_keypoints).astype(np.float32).astype(np.float64)
    if left.shape[0] == 0:
        return np.zeros((0, 3))
    uL = undistort_points(left, stereo.left_camera, round_to_f32=True)
    uR = undistort_points(right, stereo.right_camera, round_to_f32=True)
    if optimal_correction:
        uL, uR = correct_matches(stereo.F, uL, uR, round_to_f32=True)            # camera_utils.py:100-101
    P1, P2 = stereo.projection_matrices()
    points = torch.stack([uL, uR], dim=1)
    X = triangulate(points, np.stack([P1, P2]))
    return X.cpu().numpy()


class TriangulationComponent:
    """The component test/test_pipeline.py:171-177 uses: ``reset(stereo_camera)`` then
    ``__call__(left[N,2], right[N,2])`` -> [N,3] points in the left camera frame."""
    name = "triangulation"

    def __init__(self, optimal_correction=True):
        self.optimal_correction = optimal_correction
        self.stereo_camera = None

    def reset(self, stereo_camera):
        self.stereo_camera = stereo_camera

    def __call__(self, left_keypoints, right_keypoints):
        return triangulate_stereo(self.stereo_camera, left_keypoints, right_keypoints,
                                  optimal_correction=self.optimal_correction)


STEREO_ASSOCIATIONS = ('epipolar', 'depth')
DEFAULT_MAX_DEPTH_PX = 8.0      # DESIGN.md section 3: admits a +-25 % depth error at z >= 0.5 m on the ZED Mini rig


def triangulate_stereo_objects(tables, stereo, pairs=None, max_distance_px=2.5, optimal_correction=True, stream=None,
                               association='epipolar', max_depth_px=DEFAULT_MAX_DEPTH_PX):
    """The decoded objects of stereo frame pairs, matched across the two views and triangulated, on the device
    (okp_triangulate_stereo_objects_f64). tables: the DecodeTables of a batch that holds both views of every pair (decode
    it with ``camera_table((stereo.left_camera, stereo.right_camera), ...)`` so that each view is lifted with its own
    camera). pairs: [P, 2] host integers (left frame, right frame), checked here (ValueError for a bad shape,
    non-integers or frames outside the batch); None = (2p, 2p + 1), the interleaved layout, left views in even rows.
    Per pair: objects are matched by the epipolar distance of their undistorted centres, greedily one to one while it is
    <= max_distance_px (AssociationComponent's rule), then each matched object pair's slots type by type; every matched
    keypoint pair is triangulated like StereoCamera.triangulate (optimal_correction: the Hartley-Sturm correction).
    association='depth' (okp_triangulate_stereo_objects_depth_f64) tells apart objects on one epipolar line, such as
    parts side by side in the same image rows: each keypoint's lift (kp_point) is projected into the other view, and the
    greedy step runs on the mean distance d between those predictions and the other view's keypoints, over the
    candidates within max_distance_px of the epipolar line and with d <= max_depth_px. It needs lifts taken at the right
    pixel: ValueError when the tables were decoded with compat_clip_bug and a camera's image is not square.
    Returns StereoTables on the tables' device: object_match, object_cost (d with association='depth'), slot_match,
    point (left camera frame, NaN where nothing is matched), flags (_abi.STEREO_AMBIGUOUS, _abi.STEREO_BAD_PAIR,
    _abi.STEREO_NO_DEPTH). Asynchronous: nothing synchronises."""
    if association not in STEREO_ASSOCIATIONS:
        raise ValueError(f"association must be one of {STEREO_ASSOCIATIONS}, got {association!r}")
    if association == 'depth':
        sizes = [np.asarray(c.image_size).reshape(-1)[:2] for c in (stereo.left_camera, stereo.right_camera)]
        if tables.params.compat_clip_bug and any(s[0] != s[1] for s in sizes):
            raise ValueError("association='depth' reads kp_point, and with compat_clip_bug a non-square image is lifted with "
                             "the depth of a clipped column: decode with compat_clip_bug=False")
    N = tables.N
    device = tables.flat.device
    if pairs is None:
        if N % 2:
            raise ValueError(f"the interleaved layout needs an even number of frames, the tables hold {N}")
        pairs_dev = torch.arange(N, dtype=torch.int32, device=device).reshape(-1, 2)
    else:
        pairs_dev = torch.from_numpy(_abi.check_pairs(pairs, N)).to(device)
    P = int(pairs_dev.shape[0])
    O, C, S = (int(v) for v in tables['kp_xy'].shape[1:4])
    out = StereoTables(P, O, C, S, device)
    cfg = (ctypes.c_int32 * max(len(tables.keypoint_config), 1))(*tables.keypoint_config)
    left, right = _abi.pack_camera(stereo.left_camera), _abi.pack_camera(stereo.right_camera)
    F, P_L, P_R = (np.ascontiguousarray(m, dtype=np.float64) for m in (stereo.F, *stereo.projection_matrices()))
    doubles = ctypes.POINTER(ctypes.c_double)
    head = (ctypes.byref(tables.struct), N, C, cfg, ctypes.byref(tables.params), pairs_dev.data_ptr(), P, ctypes.byref(left),
            ctypes.byref(right), F.ctypes.data_as(doubles), P_L.ctypes.data_as(doubles), P_R.ctypes.data_as(doubles))
    with torch.cuda.device(device):
        if association == 'depth':
            name = 'okp_triangulate_stereo_objects_depth_f64'
            T_RL = np.ascontiguousarray(stereo.T_RL, dtype=np.float64).reshape(16)
            rc = _lib.lib().okp_triangulate_stereo_objects_depth_f64(
                *head, T_RL.ctypes.data_as(doubles), float(max_distance_px), float(max_depth_px),
                int(bool(optimal_correction)), ctypes.byref(out.struct), _stream_handle(stream))
        else:
            name = 'okp_triangulate_stereo_objects_f64'
            rc = _lib.lib().okp_triangulate_stereo_objects_f64(
                *head, float(max_distance_px), int(bool(optimal_correction)), ctypes.byref(out.struct), _stream_handle(stream))
    _lib.check(rc, name)
    out.pairs = pairs_dev                                 # the launch reads it: kept alive with the result
    return out
