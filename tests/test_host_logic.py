"""Host-side mirror of the reference interface (camera classes, linalg, synthetic generator)."""
import json
import os

import numpy as np

from object_keypoints_b200 import camera_utils, linalg, synthetic
from helpers import GOLDEN, INPUTS, load_golden, sha256

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CALIBRATION = os.path.join(ROOT, 'config', 'calibration.yaml')


def test_calibration_loading_matches_reference_semantics():
    params = camera_utils.load_calibration_params(CALIBRATION)
    cam = camera_utils.from_calibration(CALIBRATION)
    assert isinstance(cam, camera_utils.FisheyeCamera)
    assert list(cam.image_size) == [720, 1280]
    np.testing.assert_allclose(cam.K, params['K'])
    np.testing.assert_allclose(params['T_LR'] @ params['T_RL'], np.eye(4), atol=1e-12)
    g = load_golden('geometry.npz')
    np.testing.assert_array_equal(params['K'], g['K_left'])
    np.testing.assert_array_equal(params['Kp'], g['K_right'])
    np.testing.assert_array_equal(params['T_RL'], g['T_RL'])


def test_scale_and_cut_follow_eval_model_recipe():
    g = load_golden('geometry.npz')
    cam = synthetic.default_camera((64, 64))
    np.testing.assert_allclose(cam.K, g['K_net'], rtol=0, atol=1e-12)
    np.testing.assert_allclose(cam.image_size, g['image_size_net'], rtol=0, atol=1e-9)
    small = synthetic.default_camera((180, 320))
    np.testing.assert_allclose(small.K, g['K_small'], rtol=0, atol=1e-12)


def test_stereo_camera_fundamental_matrix():
    g = load_golden('geometry.npz')
    stereo = camera_utils.StereoCamera.from_file(CALIBRATION)
    np.testing.assert_allclose(stereo.F, g['F'], rtol=1e-12, atol=1e-18)
    P1, P2 = stereo.projection_matrices()
    np.testing.assert_allclose(P1, g['P1'])
    np.testing.assert_allclose(P2, g['P2'])
    # epipolar constraint on noise-free projections
    X = g['X'][:16]
    xl = stereo.left_camera.undistort(stereo.left_camera.project(X))
    xr = stereo.right_camera.undistort(stereo.right_camera.project(X, stereo.T_RL))
    hl = np.concatenate([xl, np.ones((16, 1))], axis=1)
    hr = np.concatenate([xr, np.ones((16, 1))], axis=1)
    residual = np.einsum('ni,ij,nj->n', hr, stereo.F, hl)
    scale = np.abs(stereo.F).max() * 1280 * 1280
    assert np.abs(residual).max() < 1e-9 * scale


def test_linalg():
    rng = np.random.default_rng(0)
    from scipy.spatial.transform import Rotation
    T = np.eye(4)
    T[:3, :3] = Rotation.from_rotvec(rng.normal(size=3)).as_matrix()
    T[:3, 3] = rng.normal(size=3)
    np.testing.assert_allclose(linalg.inv_transform(T) @ T, np.eye(4), atol=1e-12)
    p = rng.normal(size=(5, 3))
    np.testing.assert_allclose(linalg.transform_points(T, p), p @ T[:3, :3].T + T[:3, 3])
    v = rng.normal(size=3)
    np.testing.assert_allclose(linalg.skew_matrix(v) @ p[0], np.cross(v, p[0]))


def test_in_frame_and_unproject():
    cam = synthetic.default_camera((64, 64))
    assert list(cam.in_frame(np.array([[10.0, 10.0], [0.0, 5.0], [70.0, 5.0]]))) == [True, False, False]
    xy = np.array([[cam.K[0, 2], cam.K[1, 2]]])
    np.testing.assert_allclose(cam.unproject(xy, np.array([2.0])), [[0, 0, 2.0]], atol=1e-12)


def test_config_files():
    for name, want in (('valve.json', [1, 3]), ('cups.json', [1, 1, 1])):
        with open(os.path.join(ROOT, 'config', name)) as f:
            assert json.load(f)['keypoint_config'] == want


def test_synthetic_generator_is_deterministic_and_separated():
    a = synthetic.make_batch(3, [1, 3], (64, 64), seed=42, objects=(1, 2))
    b = synthetic.make_batch(5, [1, 3], (64, 64), seed=42, objects=(1, 2))
    np.testing.assert_array_equal(a.heat, b.heat[:3])               # per-frame substreams
    assert a.heat.dtype == np.float32 and a.heat.min() >= 0 and a.heat.max() <= 1
    assert a.centers.shape == (3, 2, 2, 64, 64) and a.depth.shape == (3, 3, 64, 64)
    for scene in a.scenes:
        if len(scene.centers) > 1:
            d = np.linalg.norm(scene.centers[0] - scene.centers[1])
            assert d >= 22.0
    # the golden fixture was produced by this very generator (it keeps the SHA-256 of the maps it was made from)
    g = np.load(os.path.join(GOLDEN, 'valve_64.npz'))
    again = synthetic.make_batch(48, [1, 3], (64, 64), seed=1001, objects=(1, 2))
    for k in INPUTS:
        assert sha256(getattr(again, k)[g['source_frames']]) == str(g['sha256_' + k]), k


def test_decode_tables_are_views_into_one_allocation():
    """DecodeTables: every table 256-byte aligned inside one buffer, numpy() = one copy with the right dtypes."""
    import torch
    from object_keypoints_b200 import _abi
    from object_keypoints_b200.pipeline import DecodeTables
    params = _abi.make_params()
    t = DecodeTables(5, 3, [1, 3], params, torch.device('cpu'))
    base = t.flat.data_ptr()
    shapes = {name: tuple(shape) for name, _, shape in _abi.table_shapes(5, 3, [1, 3], params)}
    for name, tensor in t.tensors.items():
        assert (tensor.data_ptr() - base) % DecodeTables.ALIGN == 0 and tensor.is_contiguous()
        assert tuple(tensor.shape) == shapes[name]
        assert getattr(t.struct, name) == tensor.data_ptr()
    t['kp_point'][2, 1, 0, 0, 1] = 3.5
    t['flags'][4] = 7
    t['peak_yx'][1, 2, 3, 1] = -1
    host = t.numpy()
    assert host['kp_point'][2, 1, 0, 0, 1] == 3.5 and host['kp_point'].dtype == np.float64
    assert host['flags'][4] == 7 and host['flags'].dtype == np.uint32
    assert host['peak_yx'][1, 2, 3, 1] == -1 and host['peak_xy'].dtype == np.float32
    empty = DecodeTables(0, 3, [1, 3], params, torch.device('cpu'))
    assert empty.numpy()['n_objects'].shape == (0,)


def test_bench_arms_share_one_config_and_rank_independent_step_counts():
    """bench.py: both arms print the same `config` object (the driver's same_config check), and nothing that decides how many
    exchange steps a rank runs depends on rank-local measurements (a rank-local count once deadlocked the 8-GPU run)."""
    import ast
    import inspect
    import os
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    for workload in bench.WORKLOADS:
        assert bench.workload_config(workload, 8, 'gather') == bench.workload_config(workload, 8, 'gather')
    source = inspect.getsource(bench.run_ours)
    tree = ast.parse(source)
    counts = [node for node in ast.walk(tree) if isinstance(node, ast.Assign) and
              any(isinstance(t, ast.Name) and t.id == 'count' for t in node.targets)]
    assert counts, "the sustained block's step count is gone"
    for node in counts:
        names = {n.id for n in ast.walk(node.value) if isinstance(n, ast.Name)}
        assert names <= {'max', 'args'}, f"sustained step count depends on {names - {'max', 'args'}}"


def test_sparse_auto_looks_at_the_ranks_per_host(monkeypatch):
    from object_keypoints_b200 import pipeline
    monkeypatch.setenv('LOCAL_WORLD_SIZE', '8')
    assert pipeline._local_world() == 8 and pipeline._local_world() > pipeline.KeypointDecoder.SPARSE_MAX_LOCAL_WORLD
    monkeypatch.setenv('LOCAL_WORLD_SIZE', '2')
    assert pipeline._local_world() <= pipeline.KeypointDecoder.SPARSE_MAX_LOCAL_WORLD


def test_bench_parity_rule_sees_a_single_wrong_value():
    """bench.py refuses to print a line unless every timed frame equals the oracle: the comparison itself, on oracle tables."""
    import os
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    from object_keypoints_b200 import synthetic
    from oracle import c_oracle
    cfg, size = [1, 3], (64, 64)
    batch = synthetic.make_batch(6, cfg, size, seed=4, objects=(1, 2))
    want = c_oracle.decode(batch.heat, batch.depth, batch.centers, cfg, synthetic.default_camera(size))
    assert bench.parity_mismatches(want, want) == (6, 0)
    for key, change in (('peak_yx', 1), ('kp_xy', None), ('kp_point', 1e-3), ('flags', 1)):     # None: one float32 ulp
        got = {k: v.copy() for k, v in want.items()}
        flat = got[key].reshape(6, -1)
        column = int(np.argmax(np.abs(want[key].reshape(6, -1)[2]) > 0)) if key != 'flags' else 0
        flat[2, column] = np.nextafter(flat[2, column], np.float32(np.inf)) if change is None else \
            flat[2, column] + np.asarray(change, dtype=flat.dtype)
        assert bench.parity_mismatches(got, want) == (6, 1), key


def test_bench_dump_is_exact_float_and_bounded(tmp_path):
    """bench.py --dump-outputs: every table as float32 / float64 holding exactly the decoded values, and beyond the byte
    budget the same seeded sample of frames on every run."""
    import os
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    from oracle import c_oracle
    cfg, size = [1, 3], (64, 64)
    batch = synthetic.make_batch(6, cfg, size, seed=4, objects=(1, 2))
    want = c_oracle.decode(batch.heat, batch.depth, batch.centers, cfg, synthetic.default_camera(size))
    bench.dump_outputs(str(tmp_path / 'all'), want)
    for key, value in want.items():
        got = np.load(tmp_path / 'all' / f'{key}.npy')
        assert got.dtype in (np.float32, np.float64) and got.shape == value.shape, key
        assert np.array_equal(got.astype(value.dtype), value, equal_nan=value.dtype.kind == 'f'), key
    per_frame = sum(v[0].size * (4 if v.dtype == np.float32 else 8) for v in want.values())
    for run in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / run), want, budget=3 * per_frame)
    frames = np.load(tmp_path / 'a' / 'frame_index.npy')
    assert len(frames) == 3 and np.array_equal(frames, np.load(tmp_path / 'b' / 'frame_index.npy'))
    np.testing.assert_array_equal(np.load(tmp_path / 'a' / 'kp_point.npy'), want['kp_point'][frames.astype(int)])
