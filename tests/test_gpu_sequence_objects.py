"""Sequence objects: SequenceTriangulator.objects and okp_triangulate_sequence_objects_f64. Each anchor frame's decoded
objects are matched into its view frames (by epipolar distance, or by where each frame's depth lift lands in the other
frame) and every anchor slot is triangulated over its track of V views in the world frame. The statement of record is
oracle/sequence_objects_oracle.sequence_objects (parity with the reference unpinned for V > 2, as for the per-peak chain).
CPU: the oracle against the construction, the host refusals and the Python errors. GPU: the CUDA chain against the oracle
on the same decoded tables -- matches, flags, tracks, masks and drop counts bit-equal, points <= 1e-4 relative."""
import ctypes

import numpy as np
import pytest
import torch

from helpers import TOL_METRES_REL
from object_keypoints_b200 import _abi, _lib

gpu = pytest.mark.gpu
DTYPES = {'f32': torch.float32, 'bf16': torch.bfloat16, 'f16': torch.float16}
CFG = [1, 3]
SIZE = (180, 320)
_SCENES = {}


def _scene(n_frames, noise=0.0, depth_error=0.0):
    """(camera, sequence, keypoints [N,G,Kp,2], depths [N,G,Kp], per-frame depth factors [N]), cached. The keypoints carry
    Gaussian noise of `noise` px; every frame's depth maps are to be scaled by its factor in [1 - depth_error,
    1 + depth_error]."""
    from object_keypoints_b200 import sequence, synthetic
    key = (n_frames, noise, depth_error)
    if key not in _SCENES:
        camera = synthetic.default_camera(SIZE)
        seq = sequence.synthetic_sequence(n_frames)
        keypoints, depths = sequence.project_sequence(seq, camera)
        rng = np.random.default_rng(3)
        noisy = keypoints + rng.normal(0.0, noise, keypoints.shape)
        factors = 1.0 + rng.uniform(-depth_error, depth_error, n_frames)
        _SCENES[key] = camera, seq, keypoints, noisy, depths, factors
    return _SCENES[key]


# In the wide 180x320 view a keypoint's lift reads the depth at its undistorted pixel, which lies more than 3.5 px from
# the disc drawn around its distorted pixel for about 15 % of this sequence's keypoints: wider discs give them a depth.
CENTER_RADIUS = 8.0


def _oracle_tables(n_frames, noise, depth_error):
    """The scene rasterised and decoded by the C oracle (compat_clip_bug off: the lifts are read at the right pixel)."""
    from oracle import c_oracle, np_oracle
    camera, seq, keypoints, noisy, depths, factors = _scene(n_frames, noise, depth_error)
    heat = np.zeros((n_frames, 3) + SIZE, np.float32)
    depth = np.zeros_like(heat)
    centers = np.zeros((n_frames, 2, 2) + SIZE, np.float32)
    for n in range(n_frames):
        heat[n], centers[n], depth[n] = np_oracle.rasterise_targets(noisy[n], depths[n], CFG, SIZE, center_radius=CENTER_RADIUS)
        depth[n] *= np.float32(factors[n])
    return c_oracle.decode(heat, depth, centers, CFG, camera, compat_clip_bug=False)


def _oracle(t, prepared, camera, association, **kwargs):
    from oracle import sequence_objects_oracle
    host = {k: (v.cpu().numpy() if torch.is_tensor(v) else v) for k, v in prepared.items()}
    return sequence_objects_oracle.sequence_objects(t['n_objects'], t['kp_count'], t['kp_xy'], t['kp_point'], CFG,
                                                    host['frames'], host['F'], host['motion'], host['poses'], camera,
                                                    association=association, **kwargs)


def _prepare(camera, T_CW, views):
    """SequenceTriangulator.prepare on the host (device='cpu' is enough for the oracle)."""
    from object_keypoints_b200 import sequence
    chain = sequence.SequenceTriangulator.__new__(sequence.SequenceTriangulator)
    chain.camera, chain.views, chain.device = camera, views, torch.device('cpu')
    return chain.prepare(T_CW)


def _wrong_object_matches(t, got, keypoints, frames):
    """Object matches whose two objects are different scene objects, each identified by the nearest projected centre."""
    def scene_object(f, o):
        return int(np.linalg.norm(keypoints[f, :, 0] - t['kp_xy'][f, o, 0, 0], axis=1).argmin())
    wrong = total = 0
    for a, v, o in zip(*np.nonzero(got['object_match'] >= 0)):
        total += 1
        wrong += scene_object(frames[a, 0], o) != scene_object(frames[a, v + 1], got['object_match'][a, v, o])
    return wrong, total


def _point_errors(got, seq):
    ok = ~np.isnan(got['point'][..., 0])
    truth = seq['scene'].reshape(-1, 3)
    return np.linalg.norm(got['point'][ok][:, None] - truth[None], axis=2).min(axis=1)


# ---------------------------------------------------------------------------------------------------------------------
# Host checks (no GPU)
# ---------------------------------------------------------------------------------------------------------------------
def test_prepare_forms_the_pair_motions_of_the_stereo_depth_rule():
    """motion [A,V-1,2,12] holds (R, t) of T_CW[view] inv(T_CW[anchor]) and its inverse bit for bit as the stereo depth
    oracle forms them from that matrix, next to the existing keys."""
    from object_keypoints_b200 import linalg, sequence
    from oracle.stereo_depth_oracle import _rigid
    camera, seq = _scene(24)[:2]
    prepared = _prepare(camera, seq['T_CW'], 4)
    assert {'frames', 'poses', 'F', 'frames_i32', 'motion', 'n_frames'} <= set(prepared) and prepared['n_frames'] == 24
    frames = sequence.view_schedule(24, 4)
    np.testing.assert_array_equal(prepared['frames_i32'].numpy(), frames)
    motion = prepared['motion'].numpy()
    for a in range(frames.shape[0]):
        for v in range(1, 4):
            T = seq['T_CW'][frames[a, v]] @ linalg.inv_transform(seq['T_CW'][frames[a, 0]])
            for w, (R, t) in enumerate(_rigid(T)):
                assert motion[a, v - 1, w].tobytes() == np.concatenate([R.reshape(9), t]).tobytes()


@pytest.mark.parametrize('association', ['epipolar', 'depth'])
def test_oracle_recovers_the_construction(association):
    """Noiseless 32-frame sequence, 4 views: every anchor object is matched to the same scene object in every view, and
    every anchor keypoint is triangulated within a few millimetres."""
    from object_keypoints_b200 import sequence
    camera, seq, keypoints = _scene(32)[:3]
    t = _oracle_tables(32, 0.0, 0.0)
    assert (t['n_objects'] == 8).all()
    prepared = _prepare(camera, seq['T_CW'], 4)
    got = _oracle(t, prepared, camera, association)
    frames = sequence.view_schedule(32, 4)
    wrong, total = _wrong_object_matches(t, got, keypoints, frames)
    assert wrong == 0 and total == 8 * 8 * 3
    error = _point_errors(got, seq)
    assert len(error) == 8 * 8 * 5 and np.median(error) < 2e-3 and error.max() < 1e-2
    assert not (got['flags'] & _abi.STEREO_BAD_PAIR).any()
    objects = sequence.anchor_objects(got, 0)
    assert len(objects) == 8 and [len(k) for k in objects[0]['keypoints']] == [1, 1, 3]
    assert objects[0]['p_W'][2].shape == (3, 3)


def test_depth_mode_resolves_the_objects_the_epipolar_mode_mixes_up():
    """96 frames, 8 views, keypoints with 0.3 px noise and each frame's depth maps off by up to +-10 %: the centre-epipolar
    rule matches some objects to the wrong valve (two valves on one epipolar line), the depth rule to none."""
    from object_keypoints_b200 import sequence
    camera, seq, keypoints = _scene(96, 0.3, 0.1)[:3]
    t = _oracle_tables(96, 0.3, 0.1)
    prepared = _prepare(camera, seq['T_CW'], 8)
    frames = sequence.view_schedule(96, 8)
    epipolar = _oracle(t, prepared, camera, 'epipolar')
    depth = _oracle(t, prepared, camera, 'depth')
    wrong_epipolar, _ = _wrong_object_matches(t, epipolar, keypoints, frames)
    wrong_depth, total = _wrong_object_matches(t, depth, keypoints, frames)
    assert wrong_epipolar > 0 and wrong_depth == 0 and total >= 0.99 * 12 * 7 * 8
    assert depth['dropped'].sum() < epipolar['dropped'].sum()
    assert np.median(_point_errors(depth, seq)) < 2e-3


def test_entry_validates_its_arguments_on_the_host():
    """Refusals before any CUDA call (the fake device pointers are never dereferenced)."""
    from object_keypoints_b200 import synthetic
    if _lib.needs_build():
        _lib.build()
    lib = _lib.lib()
    fake = ctypes.c_void_p(1 << 20)
    tables = _abi.OkpDecodeTables(n_objects=fake, kp_count=fake, kp_xy=fake, kp_point=fake)
    out = _abi.OkpSequenceObjectTables(**{name: fake for name, _, _ in _abi.SEQUENCE_LAYOUT})
    camera = _abi.pack_camera(synthetic.default_camera(SIZE))

    def call(tables=tables, N=32, C=2, cfg=(3,), prm=_abi.make_params(), frames=fake, A=8, V=4, F=fake, motion=fake,
             poses=fake, cam=camera, association=1, max_depth=16.0, rounds=4, out=out):
        return lib.okp_triangulate_sequence_objects_f64(
            ctypes.byref(tables) if tables is not None else None, N, C, (ctypes.c_int32 * len(cfg))(*cfg) if cfg else None,
            ctypes.byref(prm) if prm is not None else None, frames, A, V, F, motion, poses,
            ctypes.byref(cam) if cam is not None else None, association, 2.5, max_depth, 2.0, rounds,
            ctypes.byref(out) if out is not None else None, None)
    assert call(A=0, tables=None, out=None, frames=None, V=1, max_depth=-1.0) == 0                # OKP_OK: nothing to do
    for kwargs in ({'tables': None}, {'prm': None}, {'cfg': None}, {'frames': None}, {'F': None}, {'poses': None},
                   {'cam': None}, {'out': None}, {'motion': None},
                   {'tables': _abi.OkpDecodeTables(n_objects=fake, kp_count=fake, kp_xy=fake)},
                   {'tables': _abi.OkpDecodeTables(n_objects=fake, kp_count=fake, kp_point=fake)},
                   {'out': _abi.OkpSequenceObjectTables(**{name: fake for name, _, _ in _abi.SEQUENCE_LAYOUT[:-1]})}):
        assert call(**kwargs) == -1, kwargs                                                       # OKP_E_NULL
    for kwargs in ({'N': -1}, {'A': -1}, {'C': 0}, {'C': 17}, {'V': 1}, {'V': 65}, {'A': 65536}, {'rounds': -1},
                   {'prm': _abi.make_params(max_objects=65)}, {'C': 10, 'cfg': (8,) * 9},
                   {'max_depth': 0.0}, {'max_depth': -1.0}, {'max_depth': float('nan')}, {'max_depth': float('inf')},
                   {'prm': _abi.make_params(max_objects=64), 'C': 9, 'cfg': (8,) * 7 + (7,)}):            # 1 + sum = 64
        assert call(**kwargs) == -2, kwargs                                                       # OKP_E_SHAPE
    assert call(cfg=(9,)) == -3                                                                   # OKP_E_CAPACITY
    assert call(association=2) == -4 and call(association=-1) == -4                             # OKP_E_UNSUPPORTED
    # the epipolar mode reads neither the motions nor the lifts (the fake pointers would be launched on there, so only
    # the arithmetic of the shared-memory limit is checked)
    smem = lambda O, C, P: 8 * (8 * O * P + O * O + 64) + O * P + O + 2 * O * C                      # noqa: E731
    assert smem(64, 9, 64) > 227 * 1024 >= max(smem(64, 5, 32), smem(32, 9, 64))


def test_result_tables_follow_the_c_record():
    """SequenceObjectTables: every OkpSequenceObjectTables field, in its order, with its dtype and shape, in one allocation."""
    from object_keypoints_b200 import SequenceObjectTables
    tables = SequenceObjectTables(3, 4, 16, 3, 3, 'cpu')
    assert [name for name, _ in _abi.OkpSequenceObjectTables._fields_] == list(tables.tensors)
    host = tables.numpy()
    assert host['observations'].shape == (3, 16, 3, 3, 4, 2) and host['valid'].dtype == np.uint8
    assert host['object_match'].shape == (3, 3, 16) and host['flags'].dtype == np.uint32
    assert all(getattr(tables.struct, name) == tensor.data_ptr() for name, tensor in tables.tensors.items())


def test_python_refuses_unknown_modes_other_sequences_and_the_clip_quirk():
    from object_keypoints_b200 import DecodeTables, sequence
    camera, seq = _scene(24)[:2]
    chain = sequence.SequenceTriangulator.__new__(sequence.SequenceTriangulator)
    chain.camera = camera
    prepared = _prepare(camera, seq['T_CW'], 4)
    tables = DecodeTables(24, 3, CFG, _abi.make_params(), 'cpu')                        # refused before any device work
    with pytest.raises(ValueError, match='association'):
        chain.objects(tables, prepared, association='nearest')
    with pytest.raises(ValueError, match='frames'):
        chain.objects(DecodeTables(20, 3, CFG, _abi.make_params(), 'cpu'), prepared)
    with pytest.raises(ValueError, match='compat_clip_bug'):
        chain.objects(tables, prepared, association='depth')


# ---------------------------------------------------------------------------------------------------------------------
# GPU checks
# ---------------------------------------------------------------------------------------------------------------------
_MAPS = {}


def _maps(n_frames, noise, depth_error):
    """The scene rasterised on the GPU with each frame's depth factor applied, cached."""
    from object_keypoints_b200 import targets
    key = (n_frames, noise, depth_error)
    if key not in _MAPS:
        camera, seq, keypoints, noisy, depths, factors = _scene(n_frames, noise, depth_error)
        heat, depth, centers = targets.rasterise_targets(noisy, depths, CFG, SIZE, center_radius=CENTER_RADIUS)
        depth *= torch.from_numpy(factors.astype(np.float32)).cuda()[:, None, None, None]
        _MAPS[key] = heat, depth, centers
    return _MAPS[key]


def _assert_matches_oracle(got, want, what=''):
    for name in ('object_match', 'slot_match', 'flags', 'observations', 'observed', 'valid', 'dropped'):
        np.testing.assert_array_equal(got[name], want[name], err_msg=f"{what} {name}")
    np.testing.assert_allclose(got['object_cost'], want['object_cost'], rtol=1e-9, atol=1e-12, err_msg=what)
    assert np.array_equal(np.isnan(got['point']), np.isnan(want['point'])), what
    ok = ~np.isnan(want['point'][..., 0])
    deviation = np.linalg.norm(got['point'][ok] - want['point'][ok], axis=-1) / np.linalg.norm(want['point'][ok], axis=-1)
    assert deviation.max(initial=0.0) <= TOL_METRES_REL, (what, deviation.max())
    assert np.array_equal(np.isnan(got['error']), np.isnan(want['error'])), what
    solved = ~np.isnan(want['error'])
    assert np.abs(got['error'][solved] - want['error'][solved]).max(initial=0.0) < 1e-6, what
    return deviation.max(initial=0.0)


@gpu
@pytest.mark.parametrize('views', [4, 6, 8])
@pytest.mark.parametrize('association', ['epipolar', 'depth'])
@pytest.mark.parametrize('lean', [False, True])
@pytest.mark.parametrize('dtype', list(DTYPES))
def test_sequence_objects_are_the_oracle_on_the_decoded_frames(dtype, lean, association, views):
    from object_keypoints_b200 import KeypointDecoder, sequence
    camera, seq, keypoints = _scene(96, 0.3, 0.1)[:3]
    decoder = KeypointDecoder(CFG, SIZE, camera=camera, lean_tables=lean, compat_clip_bug=False)
    tables = decoder.decode_batch(*(m.to(DTYPES[dtype]) for m in _maps(96, 0.3, 0.1)))
    chain = sequence.SequenceTriangulator(camera, views=views)
    prepared = chain.prepare(seq['T_CW'])
    got = chain.objects(tables, prepared, association=association).numpy()
    t = tables.numpy()
    want = _oracle(t, prepared, camera, association)
    deviation = _assert_matches_oracle(got, want, f"{dtype} lean={lean} {association} V={views}")
    print(f"largest relative deviation from the oracle: {deviation:.3g}")
    wrong, total = _wrong_object_matches(t, got, keypoints, sequence.view_schedule(96, views))
    assert total >= 0.95 * (96 // views) * (views - 1) * 8
    if association == 'depth':
        assert wrong == 0
    assert np.median(_point_errors(got, seq)) < 3e-3


def _fabricated(camera, zero_depth=False):
    """Two frames of one camera 0.1 m apart along its x axis and three objects at one depth, objects 0 and 1 in one image
    row (on one epipolar line of the other frame): DecodeTables with each frame's keypoints and lifts, its poses."""
    from object_keypoints_b200 import DecodeTables
    X = np.array([[-0.12, 0.0, 0.8], [0.12, 0.0, 0.8], [0.0, 0.12, 0.75]])          # centre, knob, three spokes
    X = np.repeat(X[:, None], 5, axis=1) + 0.02 * np.array([[0, 0, 0], [0, 0, -1], [1, 0, 0], [0, 1, 0], [-1, -1, 0]])[None]
    T_CW = np.stack([np.eye(4), np.eye(4)])
    T_CW[1, 0, 3] = -0.1
    t = {'n_objects': np.array([3, 3], np.int32), 'kp_count': np.zeros((2, 16, 3), np.int32),
         'kp_xy': np.zeros((2, 16, 3, 3, 2), np.float32), 'kp_point': np.zeros((2, 16, 3, 3, 3))}
    t['kp_count'][:, :3] = (1, 1, 3)
    for f in range(2):
        for name, value in (('kp_xy', camera.project(X.reshape(-1, 3), T_CW[f]).reshape(3, 5, 2)),
                            ('kp_point', X @ T_CW[f, :3, :3].T + T_CW[f, :3, 3])):
            t[name][f, :3, 0, 0], t[name][f, :3, 1, 0], t[name][f, :3, 2] = value[:, 0], value[:, 1], value[:, 2:]
    if zero_depth:
        t['kp_point'][:, 0, 0, 0] = 0.0                             # object 0's centre has no depth in either frame
    tables = DecodeTables(2, 3, CFG, _abi.make_params(compat_clip_bug=False), 'cuda')
    for name, value in t.items():
        tables[name].copy_(torch.from_numpy(value))
    return tables, t, T_CW, X


@gpu
def test_objects_on_one_epipolar_line_are_told_apart_by_depth():
    from object_keypoints_b200 import sequence, synthetic
    camera = synthetic.default_camera(SIZE)
    tables, t, T_CW, X = _fabricated(camera)
    chain = sequence.SequenceTriangulator(camera, views=2)
    prepared = chain.prepare(T_CW)
    epipolar = chain.objects(tables, prepared).numpy()
    assert epipolar['flags'][0, 0] == _abi.STEREO_AMBIGUOUS
    _assert_matches_oracle(epipolar, _oracle(t, prepared, camera, 'epipolar'))
    got = chain.objects(tables, prepared, association='depth').numpy()
    _assert_matches_oracle(got, _oracle(t, prepared, camera, 'depth'))
    assert got['flags'][0, 0] == 0
    np.testing.assert_array_equal(got['object_match'][0, 0, :3], [0, 1, 2])
    points = got['point'][0, :3]                                    # [3, C, S, 3]: centre, knob, the three spokes
    np.testing.assert_allclose(points[:, 0, 0], X[:, 0], atol=1e-4)
    np.testing.assert_allclose(points[:, 1, 0], X[:, 1], atol=1e-4)
    np.testing.assert_allclose(points[:, 2], X[:, 2:], atol=1e-4)
    objects = sequence.anchor_objects(got, 0)
    assert len(objects) == 3 and np.allclose(objects[1]['p_W'][0][0], X[1, 0], atol=1e-4)


@gpu
def test_a_centre_without_depth_is_flagged_and_left_unmatched():
    """Object 0's centre lifts zeroed in both frames: the candidate has no depth on either side, it is not matched, the pair
    gets STEREO_NO_DEPTH, the anchor's track of it has one view (NaN point); the other objects are matched as before. A
    pair naming a frame outside the tables is flagged STEREO_BAD_PAIR and matches nothing."""
    from object_keypoints_b200 import sequence, synthetic
    camera = synthetic.default_camera(SIZE)
    tables, t, T_CW, X = _fabricated(camera, zero_depth=True)
    chain = sequence.SequenceTriangulator(camera, views=2)
    prepared = chain.prepare(T_CW)
    got = chain.objects(tables, prepared, association='depth').numpy()
    _assert_matches_oracle(got, _oracle(t, prepared, camera, 'depth'))
    assert got['flags'][0, 0] == _abi.STEREO_NO_DEPTH
    np.testing.assert_array_equal(got['object_match'][0, 0, :3], [-1, 1, 2])
    assert np.isnan(got['point'][0, 0]).all() and got['observed'][0, 0, 0, 0].tolist() == [1, 0]
    assert not np.isnan(got['point'][0, 1:3, 0, 0]).any()
    bad = dict(prepared, frames_i32=torch.tensor([[0, 5]], dtype=torch.int32, device='cuda'))
    got = chain.objects(tables, bad, association='depth').numpy()
    assert got['flags'][0, 0] == _abi.STEREO_BAD_PAIR and (got['object_match'] == -1).all()
    assert got['observed'][0, :3, 0, 0].tolist() == [[1, 0]] * 3 and np.isnan(got['point']).all()
