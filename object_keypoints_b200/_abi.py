"""ctypes mirror of include/okp.h: structures, table shapes and packing helpers.

Pure host code (no torch, no CUDA) so that it can be unit-tested anywhere and shared by the
library loader (``_lib.py``) and by the test-side oracle wrapper.
"""
import ctypes

import numpy as np

OKP_MAX_MAPS = 16
OKP_MAX_PEAKS = 256
OKP_MAX_OBJECTS = 128
OKP_MAX_SLOTS = 8
OKP_MAX_VIEWS = 64

FLAG_PEAK_OVERFLOW = 1
FLAG_OBJECT_OVERFLOW = 2
FLAG_OUTLIER_SKIPPED = 4
FLAG_CLUSTERED = 8
FLAG_VOTE_OVERFLOW = 16
FLAG_NO_CENTERS = 32
FLAG_ARGMAX_RESOLVED = 64
FLAG_GENERIC_PATH = 128      # property of the call, not of the data: the shape / mode ran on the exact generic kernels

STEREO_AMBIGUOUS = 1         # OkpStereoTables.flags: a left object had two or more right objects within reach
STEREO_BAD_PAIR = 2          # ... a frame index of the pair is outside the batch
STEREO_NO_DEPTH = 4          # ... association='depth': a candidate within reach had no valid lift in either view

ERRORS = {0: 'OKP_OK', -1: 'OKP_E_NULL', -2: 'OKP_E_SHAPE', -3: 'OKP_E_CAPACITY',
          -4: 'OKP_E_UNSUPPORTED', -5: 'OKP_E_CUDA', -6: 'OKP_E_WORKSPACE'}


class OkpCamera(ctypes.Structure):
    _fields_ = [('fx', ctypes.c_double), ('fy', ctypes.c_double), ('cx', ctypes.c_double), ('cy', ctypes.c_double),
                ('k', ctypes.c_double * 4), ('kinv', ctypes.c_double * 9),
                ('clip_x', ctypes.c_int32), ('clip_y', ctypes.c_int32)]


class OkpDecodeParams(ctypes.Structure):
    _fields_ = [('threshold', ctypes.c_float), ('nms_size', ctypes.c_int32), ('box_sum', ctypes.c_int32),
                ('compat_clip_bug', ctypes.c_int32), ('outlier_distance', ctypes.c_double),
                ('max_peaks', ctypes.c_int32), ('max_objects', ctypes.c_int32), ('max_votes', ctypes.c_int32),
                ('kmeans_iterations', ctypes.c_int32), ('top_k', ctypes.c_int32), ('lean_tables', ctypes.c_int32),
                ('single_pass', ctypes.c_int32)]


class OkpRecordSink(ctypes.Structure):
    _fields_ = [('buffers_dev', ctypes.POINTER(ctypes.c_void_p)), ('n_buffers', ctypes.c_int32),
                ('record_bytes', ctypes.c_int32), ('first_row', ctypes.c_longlong)]


# name, numpy dtype, shape as a function of the dimension dict -- order = field order in okp.h
TABLE_LAYOUT = [
    ('peak_count', np.int32, lambda d: (d['N'], d['C'])),
    ('peak_yx', np.int32, lambda d: (d['N'], d['C'], d['K'], 2)),
    ('peak_score', np.float32, lambda d: (d['N'], d['C'], d['K'])),
    ('peak_xy', np.float32, lambda d: (d['N'], d['C'], d['K'], 2)),
    ('peak_conf', np.float32, lambda d: (d['N'], d['C'], d['K'])),
    ('peak_object', np.int32, lambda d: (d['N'], d['C'], d['K'])),
    ('peak_vote', np.float64, lambda d: (d['N'], d['C'], d['K'], 2)),
    ('n_objects', np.int32, lambda d: (d['N'],)),
    ('flags', np.uint32, lambda d: (d['N'],)),
    ('kp_assigned', np.int32, lambda d: (d['N'], d['O'], d['C'])),
    ('kp_count', np.int32, lambda d: (d['N'], d['O'], d['C'])),
    ('kp_peak', np.int32, lambda d: (d['N'], d['O'], d['C'], d['S'])),
    ('kp_xy', np.float32, lambda d: (d['N'], d['O'], d['C'], d['S'], 2)),
    ('kp_point', np.float64, lambda d: (d['N'], d['O'], d['C'], d['S'], 3)),
    ('n_votes', np.int32, lambda d: (d['N'], d['O'])),
    ('votes', np.float64, lambda d: (d['N'], d['O'], d['V'], 2)),
]


class OkpDecodeTables(ctypes.Structure):
    _fields_ = [(name, ctypes.c_void_p) for name, _, _ in TABLE_LAYOUT]


# OkpStereoTables: name, numpy dtype, shape as a function of (P, O, C, S) -- order = field order in okp.h
STEREO_LAYOUT = [
    ('object_match', np.int32, lambda P, O, C, S: (P, O)),
    ('object_cost', np.float64, lambda P, O, C, S: (P, O)),
    ('slot_match', np.int32, lambda P, O, C, S: (P, O, C, S)),
    ('point', np.float64, lambda P, O, C, S: (P, O, C, S, 3)),
    ('flags', np.uint32, lambda P, O, C, S: (P,)),
]


class OkpStereoTables(ctypes.Structure):
    _fields_ = [(name, ctypes.c_void_p) for name, _, _ in STEREO_LAYOUT]


# OkpSequenceObjectTables: name, numpy dtype, shape as a function of (A, V, O, C, S) -- order = field order in okp.h
SEQUENCE_LAYOUT = [
    ('object_match', np.int32, lambda A, V, O, C, S: (A, V - 1, O)),
    ('object_cost', np.float64, lambda A, V, O, C, S: (A, V - 1, O)),
    ('slot_match', np.int32, lambda A, V, O, C, S: (A, V - 1, O, C, S)),
    ('flags', np.uint32, lambda A, V, O, C, S: (A, V - 1)),
    ('observations', np.float64, lambda A, V, O, C, S: (A, O, C, S, V, 2)),
    ('valid', np.uint8, lambda A, V, O, C, S: (A, O, C, S, V)),
    ('observed', np.uint8, lambda A, V, O, C, S: (A, O, C, S, V)),
    ('point', np.float64, lambda A, V, O, C, S: (A, O, C, S, 3)),
    ('error', np.float64, lambda A, V, O, C, S: (A, O, C, S, V)),
    ('dropped', np.int32, lambda A, V, O, C, S: (A, O, C, S)),
]


class OkpSequenceObjectTables(ctypes.Structure):
    _fields_ = [(name, ctypes.c_void_p) for name, _, _ in SEQUENCE_LAYOUT]


def check_pairs(pairs, N):
    """Frame pairs of okp_triangulate_stereo_objects_f64: [P, 2] integers (left frame, right frame) in [0, N) -> int32
    array. The library reads the frames they name, so they are checked here, like pack_camera_table checks its indices:
    ValueError for a shape other than [P, 2], non-integers and indices outside [0, N)."""
    pairs = np.asarray(pairs)
    if pairs.ndim != 2 or pairs.shape[1] != 2:
        raise ValueError(f"pairs must be [P, 2] (left frame, right frame), got shape {pairs.shape}")
    if pairs.size and pairs.dtype.kind not in 'iu':
        raise ValueError(f"pairs must hold integers, got {pairs.dtype}")
    if pairs.size and (pairs.min() < 0 or pairs.max() >= N):
        raise ValueError(f"pairs out of range: values in [{pairs.min()}, {pairs.max()}] for {N} frames")
    return np.ascontiguousarray(pairs, dtype=np.int32)


def table_dims(N, C, keypoint_config, params):
    return {'N': int(N), 'C': int(C), 'K': int(params.max_peaks), 'O': int(params.max_objects),
            'S': max([1] + [int(v) for v in keypoint_config]), 'V': int(params.max_votes)}


def table_shapes(N, C, keypoint_config, params):
    dims = table_dims(N, C, keypoint_config, params)
    return [(name, dtype, shape(dims)) for name, dtype, shape in TABLE_LAYOUT]


def make_params(threshold=0.5, outlier_distance=20.0, max_peaks=32, max_objects=16, max_votes=16,
                compat_clip_bug=True, kmeans_iterations=16, nms_size=5, box_sum=True, top_k=0, lean_tables=False,
                single_pass=False):
    if not (1 <= max_peaks <= OKP_MAX_PEAKS):
        raise ValueError(f"max_peaks must be in [1, {OKP_MAX_PEAKS}]")
    if not (1 <= max_objects <= OKP_MAX_OBJECTS):
        raise ValueError(f"max_objects must be in [1, {OKP_MAX_OBJECTS}]")
    if nms_size not in (3, 5):
        raise ValueError("nms_size must be 3 or 5")
    if not (0 <= top_k <= max_peaks):
        raise ValueError("top_k must be in [0, max_peaks]")
    return OkpDecodeParams(threshold=threshold, nms_size=int(nms_size), box_sum=int(bool(box_sum)), top_k=int(top_k),
                           compat_clip_bug=int(bool(compat_clip_bug)),
                           outlier_distance=outlier_distance, max_peaks=max_peaks, max_objects=max_objects,
                           max_votes=max_votes, kmeans_iterations=kmeans_iterations, lean_tables=int(bool(lean_tables)),
                           single_pass=int(bool(single_pass)))


def pack_camera(camera):
    """Camera object with K, D, Kinv, image_size (camera_utils.FisheyeCamera or the reference's
    own class) -> OkpCamera. clip_x/clip_y follow DetectionToPoint.reset (pipeline.py:159-162):
    ``image_size.astype(int) - 1`` = (H-1, W-1), later applied to (x, y)."""
    K = np.asarray(camera.K, dtype=np.float64)
    D = np.asarray(camera.D, dtype=np.float64).reshape(-1)
    if D.size < 4:
        raise ValueError("equidistant model needs four distortion coefficients")
    kinv = np.asarray(getattr(camera, 'Kinv', np.linalg.inv(K)), dtype=np.float64)
    size = np.asarray(camera.image_size)
    out = OkpCamera(fx=K[0, 0], fy=K[1, 1], cx=K[0, 2], cy=K[1, 2],
                    clip_x=int(size[0]) - 1, clip_y=int(size[1]) - 1)
    for i in range(4):
        out.k[i] = float(D[i])
    for i in range(9):
        out.kinv[i] = float(kinv.reshape(-1)[i])
    return out


def pack_camera_table(cameras, camera_index):
    """Per-frame camera table of okp_decode_cameras_* / okp_group_objects_cameras_*: a short sequence of camera objects
    (as pack_camera takes them) and camera_index [N], the camera of every frame -> ctypes array of N OkpCamera whose row n
    is pack_camera(cameras[camera_index[n]]). The library reads the rows as they are, so every index is checked here:
    ValueError for an index that is not an integer, negative or out of range, or an index array that is not 1-D."""
    index = np.asarray(camera_index)
    if index.ndim != 1:
        raise ValueError(f"camera_index must be one index per frame (1-D), got shape {index.shape}")
    if index.size and index.dtype.kind not in 'iu':
        raise ValueError(f"camera_index must hold integers, got {index.dtype}")
    packed = [pack_camera(camera) for camera in cameras]
    if index.size and (index.min() < 0 or index.max() >= len(packed)):
        raise ValueError(f"camera_index out of range: values in [{index.min()}, {index.max()}] for {len(packed)} cameras")
    table = (OkpCamera * index.size)()
    for n, c in enumerate(index.tolist()):
        table[n] = packed[c]
    return table


def check_keypoint_config(keypoint_config):
    """Accepts the parsed JSON dict {'keypoint_config': [...]} (what the reference passes,
    pipeline.py:36,95) or the bare list; returns the list of ints."""
    if isinstance(keypoint_config, dict):
        keypoint_config = keypoint_config['keypoint_config']
    cfg = [int(v) for v in keypoint_config]
    if len(cfg) + 1 > OKP_MAX_MAPS:
        raise ValueError(f"at most {OKP_MAX_MAPS - 1} keypoint types")
    if any(v < 1 or v > OKP_MAX_SLOTS for v in cfg):
        raise ValueError(f"keypoint_config entries must be in [1, {OKP_MAX_SLOTS}]")
    return cfg


def mask_unspecified(tables):
    """Copies of NumPy decode tables with every slot that ``lean_tables`` leaves unspecified (include/okp.h) reset to the
    value the default mode writes there (zero / -1), so that lean tables compare one to one with cleared ones."""
    t = {k: np.array(v, copy=True) for k, v in tables.items()}
    N, C, K = t['peak_yx'].shape[:3]
    O, S, V = t['kp_peak'].shape[1], t['kp_peak'].shape[3], t['votes'].shape[2]
    valid_peak = np.arange(K)[None, None, :] < np.minimum(t['peak_count'], K)[:, :, None]
    for name, fill in (('peak_yx', -1), ('peak_score', 0), ('peak_xy', 0), ('peak_conf', 0), ('peak_object', -1), ('peak_vote', 0)):
        mask = valid_peak if t[name].ndim == 3 else valid_peak[..., None]
        t[name] = np.where(mask, t[name], np.asarray(fill, t[name].dtype))
    valid_obj = np.arange(O)[None, :] < t['n_objects'][:, None]
    t['kp_assigned'] = np.where(valid_obj[:, :, None], t['kp_assigned'], 0)
    t['kp_count'] = np.where(valid_obj[:, :, None], t['kp_count'], 0)
    valid_slot = np.arange(S)[None, None, None, :] < t['kp_count'][..., None]
    t['kp_peak'] = np.where(valid_slot, t['kp_peak'], -1)
    t['kp_xy'] = np.where(valid_slot[..., None], t['kp_xy'], np.float32(0))
    t['kp_point'] = np.where(valid_slot[..., None], t['kp_point'], 0.0)
    t['n_votes'] = np.where(valid_obj, t['n_votes'], 0)
    valid_vote = np.arange(V)[None, None, :] < t['n_votes'][..., None]
    t['votes'] = np.where(valid_vote[..., None], t['votes'], 0.0)
    return t
