"""Stereo objects with depth association: triangulate_stereo_objects(..., association='depth') and
okp_triangulate_stereo_objects_depth_f64. Candidates are scored by where each view's lift (kp_point) lands in the other
view, which tells apart objects on one epipolar line (side by side in the same image rows). The statement of record is
oracle/stereo_depth_oracle.stereo_objects_depth; the epipolar mode's is oracle/stereo_oracle.stereo_objects."""
import ctypes

import numpy as np
import pytest
import torch

from helpers import TOL_METRES_REL
from object_keypoints_b200 import _abi, _lib

gpu = pytest.mark.gpu
DTYPES = {'f32': torch.float32, 'bf16': torch.bfloat16, 'f16': torch.float16}
SIZES = {(64, 64): [1, 1, 1], (180, 320): [1, 3]}
_BATCHES = {}


def _batch(size, cfg, scene, jitter=0.0, scale=0.0):
    """(StereoCamera, StereoBatch), cached. 'same_row': two objects per pair whose centres share a row (within jitter px),
    the keypoints of one type of an object free to share a row too; 'ordinary': stereo_batch's default scenes."""
    from object_keypoints_b200 import synthetic
    key = (size, tuple(cfg), scene, jitter, scale)
    if key not in _BATCHES:
        stereo = synthetic.stereo_rig(size)
        if scene == 'same_row':
            sb = synthetic.stereo_batch(10 if size == (64, 64) else 6, cfg, size, stereo, seed=5, objects=(2, 2), same_row=True,
                                        row_jitter=jitter, slot_margin=-1.0, depth_scale=scale, max_tries=200000)
        else:
            sb = synthetic.stereo_batch(8 if size == (64, 64) else 3, cfg, size, stereo, seed=7, depth_scale=scale)
        _BATCHES[key] = stereo, sb
    return _BATCHES[key]


def _oracle(t, pairs, cfg, stereo, association='depth', optimal_correction=True):
    from oracle import np_oracle, stereo_depth_oracle, stereo_oracle
    cameras = (np_oracle.camera_dict(stereo.left_camera), np_oracle.camera_dict(stereo.right_camera),
               stereo.left_camera.K, stereo.right_camera.K, stereo.T_RL, stereo.F)
    if association == 'epipolar':
        return stereo_oracle.stereo_objects(t['n_objects'], t['kp_count'], t['kp_xy'], pairs, cfg, *cameras,
                                            optimal_correction=optimal_correction)
    return stereo_depth_oracle.stereo_objects_depth(t['n_objects'], t['kp_count'], t['kp_xy'], t['kp_point'], pairs, cfg,
                                                    *cameras, optimal_correction=optimal_correction)


def _oracle_decode(sb, stereo):
    """Both views decoded by the C oracle with their own camera (compat_clip_bug off), interleaved again."""
    from oracle import c_oracle
    b = sb.batch
    views = [c_oracle.decode(b.heat[v::2], b.depth[v::2], b.centers[v::2], b.keypoint_config, camera, compat_clip_bug=False)
             for v, camera in enumerate((stereo.left_camera, stereo.right_camera))]
    return {k: np.stack([views[0][k], views[1][k]], 1).reshape((-1,) + views[0][k].shape[1:])
            for k in ('n_objects', 'kp_count', 'kp_xy', 'kp_point')}


# ---------------------------------------------------------------------------------------------------------------------
# Host checks (no GPU)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('scale', [0.0, 0.2])
@pytest.mark.parametrize('jitter', [0.0, 0.3])
@pytest.mark.parametrize('size', list(SIZES))
def test_depth_oracle_resolves_objects_in_one_row(size, jitter, scale):
    """Two objects per pair in one image row: epipolar matching gets some of them wrong, depth association recovers the
    construction's objects, slots and points (decode noise: 64x64 stereo depth is coarse, hence the tolerance)."""
    from object_keypoints_b200 import synthetic
    cfg = SIZES[size]
    stereo, sb = _batch(size, cfg, 'same_row', jitter, scale)
    t = _oracle_decode(sb, stereo)
    pairs = np.arange(2 * len(sb.points)).reshape(-1, 2)
    assert all(t['n_objects'] == 2)
    epipolar = _oracle(t, pairs, cfg, stereo, association='epipolar')
    assert synthetic.stereo_match_errors(sb, t, epipolar)[0] > 0 and epipolar['flags'].all()
    got = _oracle(t, pairs, cfg, stereo)
    wrong_objects, wrong_slots, worst = synthetic.stereo_match_errors(sb, t, got)
    assert (wrong_objects, wrong_slots) == (0, 0)
    assert (got['slot_match'] >= 0).sum() == 2 * len(sb.points) * (1 + sum(cfg))
    assert worst < 0.15, worst
    assert not (got['flags'] & _abi.STEREO_NO_DEPTH).any()


def test_depth_options_leave_other_batches_alone():
    """same_row and depth_scale draw nothing when off; depth_scale scales each (frame, map) depth map by its own factor."""
    from object_keypoints_b200 import synthetic
    stereo = synthetic.stereo_rig((64, 64))
    plain = synthetic.stereo_batch(4, [1, 1, 1], (64, 64), stereo, seed=7)
    scaled = synthetic.stereo_batch(4, [1, 1, 1], (64, 64), stereo, seed=7, depth_scale=0.2)
    for name in ('heat', 'centers'):
        assert getattr(plain.batch, name).tobytes() == getattr(scaled.batch, name).tobytes()
    on = plain.batch.depth > 0
    ratio = scaled.batch.depth[on] / plain.batch.depth[on]
    assert 0.8 <= ratio.min() and ratio.max() <= 1.2 and ratio.std() > 0.01


def test_depth_entry_validates_its_arguments_on_the_host():
    """Every refusal of the epipolar entry, plus NULL T_RL / kp_point, a bad max_depth_px and a shape beyond the per-block
    shared memory, before any CUDA call (the fake device pointers are never dereferenced)."""
    if _lib.needs_build():
        _lib.build()
    lib = _lib.lib()
    fake = ctypes.c_void_p(1 << 20)
    tables = _abi.OkpDecodeTables(n_objects=fake, kp_count=fake, kp_xy=fake, kp_point=fake)
    out = _abi.OkpStereoTables(**{name: fake for name, _, _ in _abi.STEREO_LAYOUT})
    camera = _abi.pack_camera(_batch((64, 64), [1, 1, 1], 'ordinary')[0].left_camera)
    m = (ctypes.c_double * 16)(*range(16))

    def call(tables=tables, N=4, C=3, cfg=(1, 3), prm=_abi.make_params(), pairs=fake, P=2, cam=camera, F=m, T=m, out=out,
             max_depth=8.0):
        return lib.okp_triangulate_stereo_objects_depth_f64(
            ctypes.byref(tables) if tables is not None else None, N, C, (ctypes.c_int32 * len(cfg))(*cfg) if cfg else None,
            ctypes.byref(prm) if prm is not None else None, pairs, P, ctypes.byref(cam) if cam is not None else None,
            ctypes.byref(camera), F, m, m, T, 2.5, max_depth, 1, ctypes.byref(out) if out is not None else None, None)
    assert call(P=0, pairs=None, tables=None, out=None, T=None, max_depth=-1.0) == 0               # OKP_OK: nothing to do
    for kwargs in ({'tables': None}, {'prm': None}, {'pairs': None}, {'cam': None}, {'F': None}, {'out': None}, {'cfg': None},
                   {'T': None}, {'tables': _abi.OkpDecodeTables(n_objects=fake, kp_count=fake, kp_xy=fake)},
                   {'tables': _abi.OkpDecodeTables(n_objects=fake, kp_count=fake, kp_point=fake)},
                   {'out': _abi.OkpStereoTables(object_match=fake, object_cost=fake, slot_match=fake, point=fake)}):
        assert call(**kwargs) == -1, kwargs                                                       # OKP_E_NULL
    for kwargs in ({'P': -1}, {'N': -1}, {'C': 0}, {'C': 17}, {'prm': _abi.make_params(max_objects=65)},
                   {'C': 10, 'cfg': (8,) * 9}, {'max_depth': 0.0}, {'max_depth': -1.0}, {'max_depth': float('nan')},
                   {'max_depth': float('inf')},
                   {'prm': _abi.make_params(max_objects=64), 'C': 9, 'cfg': (8,) * 7 + (7,)}):            # 1 + sum = 64
        assert call(**kwargs) == -2, kwargs                                                       # OKP_E_SHAPE
    assert call(cfg=(1, 9)) == -3                                                                 # OKP_E_CAPACITY
    # the largest shapes that fit: O = 64 with 1 + sum(cfg) = 32, O = 32 with 1 + sum(cfg) = 64 (the fake pointers would
    # be launched on there, so only the arithmetic of the limit is checked here)
    smem = lambda O, C, P: 8 * (8 * O * P + O * O + 64) + 5 * O * P + O + 2 * O * C                   # noqa: E731
    assert smem(64, 9, 64) > 227 * 1024 >= max(smem(64, 5, 32), smem(32, 9, 64))


def test_python_refuses_unknown_modes_and_the_clip_quirk():
    from object_keypoints_b200 import DecodeTables, triangulate_stereo_objects
    stereo_square = _batch((64, 64), [1, 1, 1], 'ordinary')[0]
    stereo_wide = _batch((180, 320), [1, 3], 'ordinary')[0]
    tables = DecodeTables(4, 3, [1, 1], _abi.make_params(), 'cpu')                      # refused before any device work
    with pytest.raises(ValueError, match='association'):
        triangulate_stereo_objects(tables, stereo_square, association='nearest')
    with pytest.raises(ValueError, match='compat_clip_bug'):
        triangulate_stereo_objects(tables, stereo_wide, association='depth')


# ---------------------------------------------------------------------------------------------------------------------
# GPU checks
# ---------------------------------------------------------------------------------------------------------------------
def _decode(size, cfg, scene, dtype='f32', lean=False):
    """The batch decoded on the GPU with one camera per view and compat_clip_bug off -> (stereo, StereoBatch, tables)."""
    from object_keypoints_b200 import KeypointDecoder
    stereo, sb = _batch(size, cfg, scene)
    b = sb.batch
    decoder = KeypointDecoder(cfg, size, lean_tables=lean, compat_clip_bug=False)
    cameras = decoder.camera_table((stereo.left_camera, stereo.right_camera), np.arange(b.heat.shape[0]) % 2)
    maps = [torch.from_numpy(a).to(DTYPES[dtype]).cuda() for a in (b.heat, b.depth, b.centers)]
    return stereo, sb, decoder.decode_batch(*maps, cameras=cameras)


def _relative(got, want):
    """Largest |got - want| / |want| over the points both have (NaN in the same places)."""
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want[..., 0])
    if not ok.any():
        return 0.0
    return float((np.linalg.norm(got[ok] - want[ok], axis=-1) / np.linalg.norm(want[ok], axis=-1)).max())


def _assert_matches_oracle(got, want, what=''):
    for name in ('object_match', 'slot_match', 'flags'):
        np.testing.assert_array_equal(got[name], want[name], err_msg=f"{what} {name}")
    np.testing.assert_allclose(got['object_cost'], want['object_cost'], rtol=1e-9, atol=1e-12, err_msg=what)
    deviation = _relative(got['point'], want['point'])
    assert deviation <= TOL_METRES_REL, (what, deviation)
    return deviation


@gpu
@pytest.mark.parametrize('scene', ['same_row', 'ordinary'])
@pytest.mark.parametrize('optimal', [True, False])
@pytest.mark.parametrize('lean', [False, True])
@pytest.mark.parametrize('dtype', list(DTYPES))
@pytest.mark.parametrize('cfg', [[1, 3], [1, 1, 1]])
@pytest.mark.parametrize('size', list(SIZES))
def test_depth_tables_are_the_oracle_on_the_decoded_frames(size, cfg, dtype, lean, optimal, scene):
    from object_keypoints_b200 import synthetic, triangulate_stereo_objects
    stereo, sb, tables = _decode(size, cfg, scene, dtype, lean)
    got = triangulate_stereo_objects(tables, stereo, optimal_correction=optimal, association='depth').numpy()
    t = tables.numpy()
    want = _oracle(t, np.arange(tables.N).reshape(-1, 2), cfg, stereo, optimal_correction=optimal)
    deviation = _assert_matches_oracle(got, want, f"{size} {cfg} {dtype} lean={lean} optimal={optimal} {scene}")
    print(f"largest relative deviation from the oracle: {deviation:.3g}")
    assert (got['object_match'] >= 0).sum() >= len(sb.points)
    if scene == 'same_row':
        assert synthetic.stereo_match_errors(sb, t, got)[:2] == (0, 0)


@gpu
def test_objects_on_one_epipolar_line_are_told_apart_by_depth():
    """The fabricated tables of the epipolar test that flags them ambiguous (two objects at one depth in one image row),
    with each view's lifts in kp_point: depth association matches every object to its own and flags nothing."""
    from object_keypoints_b200 import DecodeTables, triangulate_stereo_objects
    size, cfg = (64, 64), [1, 1, 1]
    stereo = _batch(size, cfg, 'ordinary')[0]
    params = _abi.make_params()
    X = np.array([[-0.15, 0.0, 1.0], [0.15, 0.0, 1.0], [0.0, 0.2, 0.9]])                # objects 0 and 1 on one row
    X = np.repeat(X[:, None], 4, axis=1) + 0.02 * np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [-1, -1, 0]])[None]
    t = {'n_objects': np.array([3, 3], np.int32), 'kp_count': np.zeros((2, 16, 4), np.int32),
         'kp_xy': np.zeros((2, 16, 4, 1, 2), np.float32), 'kp_point': np.zeros((2, 16, 4, 1, 3))}
    t['kp_count'][:, :3] = 1
    for v, (camera, T) in enumerate(((stereo.left_camera, np.eye(4)), (stereo.right_camera, stereo.T_RL))):
        t['kp_xy'][v, :3, :, 0] = camera.project(X.reshape(-1, 3), T).reshape(3, 4, 2)
        t['kp_point'][v, :3, :, 0] = X @ T[:3, :3].T + T[:3, 3]
    tables = DecodeTables(2, 4, cfg, params, 'cuda')
    for name, value in t.items():
        tables[name].copy_(torch.from_numpy(value))
    assert triangulate_stereo_objects(tables, stereo).numpy()['flags'][0] == _abi.STEREO_AMBIGUOUS
    got = triangulate_stereo_objects(tables, stereo, association='depth').numpy()
    want = _oracle(t, np.array([[0, 1]]), cfg, stereo)
    _assert_matches_oracle(got, want)
    assert got['flags'][0] == 0
    np.testing.assert_array_equal(got['object_match'][0, :3], [0, 1, 2])
    assert _relative(got['point'][0, :3, :, 0], X) < 1e-5


@gpu
def test_a_keypoint_without_depth_is_flagged_and_left_unmatched():
    """The depth disc of one object's centre zeroed in both views: its lifts are (0, 0, 0), so the candidate has no depth
    on either side. It is not matched, the pair gets STEREO_NO_DEPTH, and the other objects are matched as before."""
    from object_keypoints_b200 import KeypointDecoder, synthetic, triangulate_stereo_objects
    size, cfg = (64, 64), [1, 1, 1]
    stereo, sb = _batch(size, cfg, 'same_row')
    b = sb.batch
    depth = b.depth.copy()
    for v, o in enumerate((0, sb.right_of_left[0][0])):                                 # one object in both views
        window, mask, _, _ = synthetic._disc(size[0], size[1], sb.pixels[0][v][o, 0])
        depth[v, 0][window][mask] = 0.0
    decoder = KeypointDecoder(cfg, size, compat_clip_bug=False)
    cameras = decoder.camera_table((stereo.left_camera, stereo.right_camera), np.arange(b.heat.shape[0]) % 2)
    tables = decoder.decode_batch(b.heat, depth, b.centers, cameras=cameras)
    got = triangulate_stereo_objects(tables, stereo, association='depth').numpy()
    t = tables.numpy()
    want = _oracle(t, np.arange(tables.N).reshape(-1, 2), cfg, stereo)
    _assert_matches_oracle(got, want)
    i = int(np.linalg.norm(t['kp_xy'][0, :2, 0, 0] - sb.pixels[0][0][0, 0], axis=-1).argmin())
    assert (t['kp_point'][0, i, 0, 0] == 0).all()
    assert got['flags'][0] == _abi.STEREO_NO_DEPTH
    assert got['object_match'][0, i] == -1 and np.isnan(got['point'][0, i]).all()
    assert (got['object_match'][0, 1 - i] >= 0) and not (got['flags'][1:] & _abi.STEREO_NO_DEPTH).any()
