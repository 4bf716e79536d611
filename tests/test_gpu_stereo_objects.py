"""Stereo objects: okp_triangulate_stereo_objects_f64 and triangulate_stereo_objects. The decoded objects of frame pairs
are matched across the two views (centres, then slots type by type) and triangulated in the left camera's frame; the
statement of record is oracle/stereo_oracle.stereo_objects, itself a composition of np_oracle.associate and
np_oracle.triangulate_stereo."""
import ctypes

import numpy as np
import pytest
import torch

from helpers import load_golden, TOL_METRES_REL
from object_keypoints_b200 import _abi, _lib

gpu = pytest.mark.gpu
DTYPES = {'f32': torch.float32, 'bf16': torch.bfloat16}
PAIRS = {(64, 64): 8, (180, 320): 3}
_BATCHES = {}


def _stereo(size, cfg, seed=7):
    """(StereoCamera, StereoBatch) of the calibration rig at the prediction size, cached."""
    from object_keypoints_b200 import synthetic
    key = (size, tuple(cfg), seed)
    if key not in _BATCHES:
        stereo = synthetic.stereo_rig(size)
        _BATCHES[key] = stereo, synthetic.stereo_batch(PAIRS[size], cfg, size, stereo, seed=seed)
    return _BATCHES[key]


def _oracle(t, pairs, cfg, stereo, max_distance_px=2.5, optimal_correction=True):
    from oracle import np_oracle, stereo_oracle
    return stereo_oracle.stereo_objects(t['n_objects'], t['kp_count'], t['kp_xy'], pairs, cfg,
                                    np_oracle.camera_dict(stereo.left_camera), np_oracle.camera_dict(stereo.right_camera),
                                    stereo.left_camera.K, stereo.right_camera.K, stereo.T_RL, stereo.F,
                                    max_distance_px, optimal_correction)


def _oracle_decode(batch, stereo):
    """Both views decoded by the C oracle with their own camera, interleaved again -> n_objects, kp_count, kp_xy."""
    from oracle import c_oracle
    cfg = batch.keypoint_config
    views = [c_oracle.decode(batch.heat[v::2], batch.depth[v::2], batch.centers[v::2], cfg, camera)
             for v, camera in enumerate((stereo.left_camera, stereo.right_camera))]
    return {k: np.stack([views[0][k], views[1][k]], 1).reshape((-1,) + views[0][k].shape[1:])
            for k in ('n_objects', 'kp_count', 'kp_xy')}


def _relative(got, want):
    """Largest |got - want| / |want| over the points both have (NaN in the same places)."""
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want[..., 0])
    if not ok.any():
        return 0.0
    return float((np.linalg.norm(got[ok] - want[ok], axis=-1) / np.linalg.norm(want[ok], axis=-1)).max())


# ---------------------------------------------------------------------------------------------------------------------
# Host checks (no GPU)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('size,cfg', [((64, 64), [1, 1, 1]), ((180, 320), [1, 3])])
def test_oracle_is_associate_and_triangulate_stereo_pair_by_pair(size, cfg):
    from oracle import np_oracle
    stereo, sb = _stereo(size, cfg)
    t = _oracle_decode(sb.batch, stereo)
    P = len(sb.points)
    got = _oracle(t, np.arange(2 * P).reshape(-1, 2), cfg, stereo)
    cl, cr = np_oracle.camera_dict(stereo.left_camera), np_oracle.camera_dict(stereo.right_camera)
    for p in range(P):
        l, r = 2 * p, 2 * p + 1

        def und(f, o, c, cam):
            return np.array([np_oracle.undistort_point(float(x), float(y), cam)
                             for x, y in t['kp_xy'][f, o, c, :t['kp_count'][f, o, c]]]).reshape(-1, 2)
        nl, nr = int(t['n_objects'][l]), int(t['n_objects'][r])
        match, cost = np_oracle.associate(stereo.F, np.array([und(l, o, 0, cl)[0] for o in range(nl)]).reshape(-1, 2),
                                          np.array([und(r, o, 0, cr)[0] for o in range(nr)]).reshape(-1, 2))
        np.testing.assert_array_equal(got['object_match'][p, :nl], match)
        np.testing.assert_array_equal(got['object_cost'][p, :nl], cost)
        assert (got['object_match'][p, nl:] == -1).all()
        for i, j in enumerate(match.tolist()):
            if j < 0:
                assert (got['slot_match'][p, i] == -1).all() and np.isnan(got['point'][p, i]).all()
                continue
            for c in range(len(cfg) + 1):
                slots = np.zeros(1, np.int32) if c == 0 else np_oracle.associate(stereo.F, und(l, i, c, cl), und(r, j, c, cr))[0]
                np.testing.assert_array_equal(got['slot_match'][p, i, c, :len(slots)], slots)
                for s, m in enumerate(slots.tolist()):
                    if m < 0:
                        continue
                    want = np_oracle.triangulate_stereo(t['kp_xy'][l, i, c, s:s + 1], t['kp_xy'][r, j, c, m:m + 1], cl, cr,
                                                        stereo.left_camera.K, stereo.right_camera.K, stereo.T_RL, stereo.F)
                    np.testing.assert_array_equal(got['point'][p, i, c, s], want[0])
        assert got['object_match'][p, :nl].max() >= 0


@pytest.mark.parametrize('size,cfg', [((64, 64), [1, 1, 1]), ((180, 320), [1, 3])])
def test_oracle_recovers_the_construction_on_noiseless_keypoints(size, cfg):
    """Tables holding the construction's own (float32) pixels: the matches are the construction's permutation and the
    points are its 3D points."""
    stereo, sb = _stereo(size, cfg)
    t = _noiseless_tables(sb, cfg)
    got = _oracle(t, np.arange(2 * len(sb.points)).reshape(-1, 2), cfg, stereo)
    assert not got['flags'].any()
    for p, (perm, X) in enumerate(zip(sb.right_of_left, sb.points)):
        n = len(perm)
        np.testing.assert_array_equal(got['object_match'][p, :n], perm)
        k = 0
        for c, count in enumerate([1] + cfg):
            np.testing.assert_array_equal(got['slot_match'][p, :n, c, :count], np.broadcast_to(np.arange(count), (n, count)))
            assert _relative(got['point'][p, :n, c, :count].reshape(-1, 3), X[:, k:k + count].reshape(-1, 3)) < 1e-5
            k += count


def _noiseless_tables(sb, cfg):
    """n_objects, kp_count, kp_xy of the construction's pixels (float32), interleaved like the batch."""
    P, O, C, S = len(sb.points), 16, 1 + len(cfg), max(cfg)
    t = {'n_objects': np.zeros(2 * P, np.int32), 'kp_count': np.zeros((2 * P, O, C), np.int32),
         'kp_xy': np.zeros((2 * P, O, C, S, 2), np.float32)}
    for p, views in enumerate(sb.pixels):
        for v, px in enumerate(views):
            f, n = 2 * p + v, px.shape[0]
            t['n_objects'][f] = n
            k = 0
            for c, count in enumerate([1] + cfg):
                t['kp_count'][f, :n, c] = count
                t['kp_xy'][f, :n, c, :count] = px[:, k:k + count]
                k += count
    return t


@pytest.mark.parametrize('pairs,match', [
    (np.array([[0, 4]]), 'range'), (np.array([[-1, 1]]), 'range'), (np.array([[0.0, 1.0]]), 'integers'),
    (np.array([0, 1]), r'\[P, 2\]'), (np.zeros((2, 3), np.int64), r'\[P, 2\]'), ([[True, False]], 'integers'),
])
def test_pairs_are_checked_on_the_host(pairs, match):
    from object_keypoints_b200 import DecodeTables, triangulate_stereo_objects
    with pytest.raises(ValueError, match=match):
        _abi.check_pairs(pairs, 4)
    tables = DecodeTables(4, 3, [1, 1], _abi.make_params(), 'cpu')          # refused before anything touches a device
    with pytest.raises(ValueError, match=match):
        triangulate_stereo_objects(tables, _stereo((64, 64), [1, 1, 1])[0], pairs=pairs)
    with pytest.raises(ValueError, match='even'):
        triangulate_stereo_objects(DecodeTables(3, 3, [1, 1], _abi.make_params(), 'cpu'), _stereo((64, 64), [1, 1, 1])[0])
    assert _abi.check_pairs(np.array([[3, 0], [1, 2]], np.uint8), 4).dtype == np.int32


def test_entry_validates_its_arguments_on_the_host():
    """NULL pointers and bad shapes are refused before any CUDA call (the fake device pointers are never dereferenced)."""
    if _lib.needs_build():
        _lib.build()
    lib = _lib.lib()
    fake = ctypes.c_void_p(1 << 20)
    tables = _abi.OkpDecodeTables(n_objects=fake, kp_count=fake, kp_xy=fake)
    out = _abi.OkpStereoTables(**{name: fake for name, _, _ in _abi.STEREO_LAYOUT})
    camera = _abi.pack_camera(_stereo((64, 64), [1, 1, 1])[0].left_camera)
    m = (ctypes.c_double * 12)(*range(12))

    def call(tables=tables, N=4, C=3, cfg=(1, 3), prm=_abi.make_params(), pairs=fake, P=2, cam=camera, F=m, out=out):
        return lib.okp_triangulate_stereo_objects_f64(
            ctypes.byref(tables) if tables is not None else None, N, C, (ctypes.c_int32 * len(cfg))(*cfg) if cfg else None,
            ctypes.byref(prm) if prm is not None else None, pairs, P, ctypes.byref(cam) if cam is not None else None,
            ctypes.byref(camera), F, m, m, 2.5, 1, ctypes.byref(out) if out is not None else None, None)
    assert call(P=0, pairs=None, tables=None, out=None) == 0                                 # OKP_OK: nothing to do
    for kwargs in ({'tables': None}, {'prm': None}, {'pairs': None}, {'cam': None}, {'F': None}, {'out': None}, {'cfg': None},
                   {'tables': _abi.OkpDecodeTables(n_objects=fake, kp_count=fake)},
                   {'out': _abi.OkpStereoTables(object_match=fake, object_cost=fake, slot_match=fake, point=fake)}):
        assert call(**kwargs) == -1, kwargs                                                 # OKP_E_NULL
    for kwargs in ({'P': -1}, {'N': -1}, {'C': 0}, {'C': 17}, {'prm': _abi.make_params(max_objects=65)},
                   {'C': 10, 'cfg': (8,) * 9}):
        assert call(**kwargs) == -2, kwargs                                                 # OKP_E_SHAPE
    assert call(cfg=(1, 9)) == -3                                                           # OKP_E_CAPACITY


# ---------------------------------------------------------------------------------------------------------------------
# GPU checks
# ---------------------------------------------------------------------------------------------------------------------
def _decode(size, cfg, dtype='f32', lean=False, seed=7):
    """The stereo batch decoded on the GPU with one camera per view -> (stereo, StereoBatch, DecodeTables)."""
    from object_keypoints_b200 import KeypointDecoder
    stereo, sb = _stereo(size, cfg, seed)
    b = sb.batch
    decoder = KeypointDecoder(cfg, size, lean_tables=lean)
    cameras = decoder.camera_table((stereo.left_camera, stereo.right_camera), np.arange(b.heat.shape[0]) % 2)
    maps = [torch.from_numpy(a).to(DTYPES[dtype]).cuda() for a in (b.heat, b.depth, b.centers)]
    return stereo, sb, decoder.decode_batch(*maps, cameras=cameras)


def _assert_matches_oracle(got, want, what=''):
    for name in ('object_match', 'slot_match', 'flags'):
        np.testing.assert_array_equal(got[name], want[name], err_msg=f"{what} {name}")
    np.testing.assert_allclose(got['object_cost'], want['object_cost'], rtol=1e-9, atol=1e-12, err_msg=what)
    deviation = _relative(got['point'], want['point'])
    assert deviation <= TOL_METRES_REL, (what, deviation)
    return deviation


@gpu
@pytest.mark.parametrize('optimal', [True, False])
@pytest.mark.parametrize('lean', [False, True])
@pytest.mark.parametrize('dtype', ['f32', 'bf16'])
@pytest.mark.parametrize('cfg', [[1, 3], [1, 1, 1]])
@pytest.mark.parametrize('size', [(64, 64), (180, 320)])
def test_tables_are_the_oracle_on_the_decoded_frames(size, cfg, dtype, lean, optimal):
    from object_keypoints_b200 import triangulate_stereo_objects
    stereo, sb, tables = _decode(size, cfg, dtype, lean)
    got = triangulate_stereo_objects(tables, stereo, optimal_correction=optimal).numpy()
    t = tables.numpy()
    want = _oracle(t, np.arange(tables.N).reshape(-1, 2), cfg, stereo, optimal_correction=optimal)
    deviation = _assert_matches_oracle(got, want, f"{size} {cfg} {dtype} lean={lean} optimal={optimal}")
    print(f"largest relative deviation from the oracle: {deviation:.3g}")
    assert (got['object_match'] >= 0).sum() >= len(sb.points) and not np.isnan(got['point'][:, :, 0, 0][got['object_match'] >= 0]).any()


@gpu
def test_reference_stereo_test_frames():
    """test/test_pipeline.py:179-206 of the reference: both views of its stereo test decoded in one call with per-frame
    cameras, then triangulated; the centre within 5e-2 m of the truth, every point TriangulationComponent's."""
    from object_keypoints_b200 import KeypointDecoder, TriangulationComponent, camera_utils, triangulate_stereo_objects
    g = load_golden('test_pipeline_180x320.npz')
    geo = load_golden('geometry.npz')
    left, right = (camera_utils.FisheyeCamera(geo[f'K_{v}'], geo[f'D_{v}'], [720, 1280]).scale(180 / 720)
                   for v in ('left', 'right'))
    stereo = camera_utils.StereoCamera(left, right, g['T_RL'])
    cfg = [int(v) for v in g['keypoint_config']]
    decoder = KeypointDecoder(cfg, (180, 320))
    tables = decoder.decode_batch(g['heat'], g['depth'], g['centers'], cameras=decoder.camera_table((left, right), [0, 1]))
    got = triangulate_stereo_objects(tables, stereo).numpy()
    t = tables.numpy()
    assert got['object_match'][0, 0] == 0 and not got['flags'].any()
    assert np.linalg.norm(got['point'][0, 0, 0, 0] - g['keypoints_3d'][0]) < 5e-2
    triangulation = TriangulationComponent()
    triangulation.reset(stereo)
    matched = 0
    for o, c, s in zip(*np.nonzero(got['slot_match'][0] >= 0)):
        j, m = got['object_match'][0, o], got['slot_match'][0, o, c, s]
        want = triangulation(t['kp_xy'][0, o, c, s:s + 1], t['kp_xy'][1, j, c, m:m + 1])[0]
        assert np.linalg.norm(got['point'][0, o, c, s] - want) <= 1e-9 * np.linalg.norm(want)
        matched += 1
    assert matched == 1 + sum(cfg)


@gpu
def test_layouts_empty_frames_and_empty_types():
    from object_keypoints_b200 import triangulate_stereo_objects
    size, cfg = (64, 64), [1, 3]
    stereo, sb, tables = _decode(size, cfg)
    N = tables.N
    interleaved = triangulate_stereo_objects(tables, stereo).numpy()
    # left views in the first half, right views in the second: the same pairs, the same tables
    order = np.concatenate([np.arange(0, N, 2), np.arange(1, N, 2)])
    blocks = type(tables)(N, tables.C, cfg, tables.params, 'cuda')
    for name, tensor in tables.tensors.items():
        blocks[name].copy_(tensor[torch.from_numpy(order).cuda()])
    got = triangulate_stereo_objects(blocks, stereo, pairs=np.stack([np.arange(N // 2), np.arange(N // 2) + N // 2], 1)).numpy()
    for name in interleaved:
        np.testing.assert_array_equal(got[name], interleaved[name], err_msg=name)
    # pair 0 without objects on the right, pair 1 without keypoints of type 1 on the left
    tables['n_objects'][1] = 0
    tables['kp_count'][2, :, 1] = 0
    got = triangulate_stereo_objects(tables, stereo).numpy()
    want = _oracle(tables.numpy(), np.arange(N).reshape(-1, 2), cfg, stereo)
    _assert_matches_oracle(got, want)
    assert (got['object_match'][0] == -1).all() and np.isnan(got['point'][0]).all() and not got['flags'][0]
    assert (got['slot_match'][1, :, 1] == -1).all() and (got['slot_match'][1, :, 2] >= 0).any()
    # no pairs
    empty = triangulate_stereo_objects(tables, stereo, pairs=np.zeros((0, 2), np.int64))
    assert empty.P == 0 and empty['point'].shape[0] == 0


@gpu
def test_a_pair_outside_the_batch_is_flagged_and_matches_nothing():
    """Python refuses such pairs; the C entry reports them per pair."""
    from object_keypoints_b200 import StereoTables
    size, cfg = (64, 64), [1, 1, 1]
    stereo, _, tables = _decode(size, cfg)
    N = tables.N
    pairs = torch.tensor([[0, 1], [0, N], [-1, 3], [2, 3]], dtype=torch.int32, device='cuda')
    out = StereoTables(4, *tables['kp_xy'].shape[1:4], 'cuda')
    out['object_match'].fill_(7)
    cfg_c = (ctypes.c_int32 * len(cfg))(*cfg)
    F, P_L, P_R = (np.ascontiguousarray(m, dtype=np.float64) for m in (stereo.F, *stereo.projection_matrices()))
    d = ctypes.POINTER(ctypes.c_double)
    rc = _lib.lib().okp_triangulate_stereo_objects_f64(
        ctypes.byref(tables.struct), N, tables.C, cfg_c, ctypes.byref(tables.params), pairs.data_ptr(), 4,
        ctypes.byref(_abi.pack_camera(stereo.left_camera)), ctypes.byref(_abi.pack_camera(stereo.right_camera)),
        F.ctypes.data_as(d), P_L.ctypes.data_as(d), P_R.ctypes.data_as(d), 2.5, 1, ctypes.byref(out.struct), None)
    assert rc == 0
    got = out.numpy()
    np.testing.assert_array_equal(got['flags'], [0, _abi.STEREO_BAD_PAIR, _abi.STEREO_BAD_PAIR, 0])
    for p in (1, 2):
        assert (got['object_match'][p] == -1).all() and (got['object_cost'][p] == 0).all()
        assert (got['slot_match'][p] == -1).all() and np.isnan(got['point'][p]).all()
    want = _oracle(tables.numpy(), pairs.cpu().numpy(), cfg, stereo)
    _assert_matches_oracle(got, want)


@gpu
def test_objects_on_one_epipolar_line_are_flagged_ambiguous():
    """Two objects at one depth and one image row: each left centre has both right centres within reach. The greedy
    step still matches one to one; the flag says the match is not determined by the geometry."""
    from object_keypoints_b200 import DecodeTables, triangulate_stereo_objects
    size, cfg = (64, 64), [1, 1, 1]
    stereo, _ = _stereo(size, cfg)
    params = _abi.make_params()
    X = np.array([[-0.15, 0.0, 1.0], [0.15, 0.0, 1.0], [0.0, 0.2, 0.9]])                # objects 0 and 1 on one row
    X = np.repeat(X[:, None], 4, axis=1) + 0.02 * np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [-1, -1, 0]])[None]
    t = {'n_objects': np.array([3, 3], np.int32), 'kp_count': np.zeros((2, 16, 4), np.int32),
         'kp_xy': np.zeros((2, 16, 4, 1, 2), np.float32)}
    t['kp_count'][:, :3] = 1
    for v, (camera, T) in enumerate(((stereo.left_camera, np.eye(4)), (stereo.right_camera, stereo.T_RL))):
        t['kp_xy'][v, :3, :, 0] = camera.project(X.reshape(-1, 3), T).reshape(3, 4, 2)
    tables = DecodeTables(2, 4, cfg, params, 'cuda')
    for name, value in t.items():
        tables[name].copy_(torch.from_numpy(value))
    got = triangulate_stereo_objects(tables, stereo).numpy()
    want = _oracle(t, np.array([[0, 1]]), cfg, stereo)
    assert want['flags'][0] == _abi.STEREO_AMBIGUOUS
    _assert_matches_oracle(got, want)
