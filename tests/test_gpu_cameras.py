"""Per-frame cameras: okp_decode_cameras_* / okp_group_objects_cameras_* and the ``cameras=`` keyword of the Python API.
Frame n of a batch is lifted with its own row of a camera table; everything but the camera is the single-camera decode's
arithmetic, so the rows of camera c must be those of a single-camera decode with camera c, bit for bit."""
import ctypes
import os

import numpy as np
import pytest
import torch

from object_keypoints_b200 import _abi, _lib
from test_gpu_decode import assert_matches_oracle
from test_gpu_f16 import _assert_same_tables

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CALIBRATION = os.path.join(ROOT, 'config', 'calibration.yaml')
CFG = [1, 3]
DTYPES = {'f32': torch.float32, 'bf16': torch.bfloat16, 'f16': torch.float16}
# Stereo scene: largest distance (m) between a left-view point and the matching right-view point mapped by T_LR. A CPU
# rehearsal with the C oracle (test_stereo_tolerance_on_the_oracle) gives 1.9 mm with each view's own camera and 8.1 mm
# with cam0 for both views.
STEREO_TOL = 4e-3


def _fit(camera, size, extra_offset=(0.0, 0.0)):
    """synthetic.default_camera's recipe for any calibrated camera: 64x64 = scale to the 511 px network input, cut to a
    square, scale to 64; other sizes = scale to the prediction height. extra_offset widens the cut."""
    if tuple(size) == (64, 64):
        scaled = camera.scale(511.0 / 720.0)
        offset = np.array([(scaled.image_size[1] - 511.0) / 2.0, 0.0]) + np.asarray(extra_offset)
        return scaled.cut(offset).scale(64.0 / 511.0)
    scaled = camera.scale(size[0] / 720.0)
    return scaled.cut(np.asarray(extra_offset)) if any(extra_offset) else scaled


def _rig():
    from object_keypoints_b200 import camera_utils
    p = camera_utils.load_calibration_params(CALIBRATION)
    return (camera_utils.FisheyeCamera(p['K'], p['D'], p['image_size']),
            camera_utils.FisheyeCamera(p['Kp'], p['Dp'], p['image_size']), p)


def _cameras(size):
    """cam0, cam1 and cam0 cut with another offset (another image_size, so another clip_x / clip_y)."""
    cam0, cam1, _ = _rig()
    third = _fit(cam0, size, (12.0, 20.0) if tuple(size) == (64, 64) else (8.0, 4.0))
    return [_fit(cam0, size), _fit(cam1, size), third]


def _index(pattern, N):
    if pattern == 'alternating':
        return np.arange(N) % 2
    if pattern == 'blocks':
        return np.minimum(np.arange(N) * 3 // N, 2)
    return np.random.default_rng(N).integers(0, 3, N)


_BATCHES = {}


def _batch(size):
    """(heat, depth, centers) float32 CPU tensors: bench-style grid frames at 180x320 (32-lane grouping), the seeded NumPy
    generator at 64x64 (16-lane grouping)."""
    if size not in _BATCHES:
        from object_keypoints_b200 import synthetic
        if size == (180, 320):
            maps = synthetic.torch_grid_batch(24, CFG, size, seed=31, grid=(4, 2), device='cuda')[:3]
            _BATCHES[size] = tuple(t.cpu() for t in maps)
        else:
            batch = synthetic.make_batch(48, CFG, size, seed=32, objects=(1, 3))
            _BATCHES[size] = tuple(torch.from_numpy(a) for a in (batch.heat, batch.depth, batch.centers))
    return _BATCHES[size]


def _maps(size, dtype):
    """-> (CUDA maps of the dtype, their float32 up-cast as NumPy for the oracle)."""
    maps = [t.to(DTYPES[dtype]).cuda() for t in _batch(size)]
    return maps, [t.float().cpu().numpy() for t in maps]


def _rows(tables, idx, lean):
    rows = {k: v[idx] for k, v in tables.items()}
    return _abi.mask_unspecified(rows) if lean else rows


# ---------------------------------------------------------------------------------------------------------------------
# GPU checks
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize('pattern', ['alternating', 'blocks', 'random'])
@pytest.mark.parametrize('lean', [False, True])
@pytest.mark.parametrize('dtype', ['f32', 'bf16', 'f16'])
@pytest.mark.parametrize('size', [(180, 320), (64, 64)])
def test_rows_of_each_camera_are_the_oracle_and_the_single_camera_decode(size, dtype, lean, pattern):
    from oracle import c_oracle
    from object_keypoints_b200 import KeypointDecoder
    cameras = _cameras(size)
    (heat, depth, centers), host = _maps(size, dtype)
    N = heat.shape[0]
    index = _index(pattern, N)
    decoder = KeypointDecoder(CFG, size, lean_tables=lean)
    table = decoder.camera_table(cameras, index)
    got = decoder.decode_batch(heat, depth, centers, cameras=table).numpy()
    for c, camera in enumerate(cameras):
        idx = np.flatnonzero(index == c)
        if idx.size == 0:
            continue
        want = c_oracle.decode(*(a[idx] for a in host), CFG, camera)
        assert_matches_oracle(_rows(got, idx, lean), _abi.mask_unspecified(want) if lean else want)
        single = KeypointDecoder(CFG, size, camera=camera, lean_tables=lean)
        sel = torch.from_numpy(idx).cuda()
        alone = single.decode_batch(heat[sel], depth[sel], centers[sel]).numpy()
        _assert_same_tables(_rows(got, idx, lean), _rows(alone, np.arange(idx.size), lean), f"camera {c}")
    assert got['n_objects'].sum() > 0 and np.abs(got['kp_point']).sum() > 0


@gpu
@pytest.mark.parametrize('lean', [False, True])
@pytest.mark.parametrize('dtype', ['f32', 'bf16', 'f16'])
@pytest.mark.parametrize('size', [(180, 320), (64, 64)])
def test_one_camera_on_every_row_is_the_reset_decode(size, dtype, lean):
    from object_keypoints_b200 import KeypointDecoder
    camera = _cameras(size)[1]
    (heat, depth, centers), _ = _maps(size, dtype)
    N = heat.shape[0]
    decoder = KeypointDecoder(CFG, size, camera=camera, lean_tables=lean)
    table = decoder.camera_table([camera], np.zeros(N, np.int64))
    want = _rows(decoder.decode_batch(heat, depth, centers).numpy(), slice(None), lean)
    got = _rows(decoder.decode_batch(heat, depth, centers, cameras=table).numpy(), slice(None), lean)
    _assert_same_tables(got, want)
    # the two-call path (peaks, then okp_group_objects_cameras_*) and KeypointDecoder.group_objects
    got = decoder.decode_batch(heat, depth, centers, cameras=table, peaks_done=torch.cuda.Event())
    _assert_same_tables(_rows(got.numpy(), slice(None), lean), want)
    decoder.group_objects(depth, centers, got, cameras=table)
    _assert_same_tables(_rows(got.numpy(), slice(None), lean), want)
    with pytest.raises(ValueError, match='rows'):
        decoder.decode_batch(heat[:N - 1], depth[:N - 1], centers[:N - 1], cameras=table)
    # a batch of no frames: nothing to do, as with one camera (the empty table's pointer is NULL)
    empty = decoder.camera_table([camera], np.zeros(0, np.int64))
    assert decoder.decode_batch(heat[:0], depth[:0], centers[:0], cameras=empty).N == 0


@gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_a_table_on_another_device_is_refused():
    from object_keypoints_b200 import KeypointDecoder
    size = (64, 64)
    camera = _cameras(size)[0]
    (heat, depth, centers), _ = _maps(size, 'f32')
    N = heat.shape[0]
    other = KeypointDecoder(CFG, size, device='cuda:1').camera_table([camera], np.zeros(N, np.int64))
    decoder = KeypointDecoder(CFG, size, camera=camera, device='cuda:0')
    with pytest.raises(ValueError, match='device|cuda:1'):
        decoder.decode_batch(heat, depth, centers, cameras=other)
    with pytest.raises(ValueError, match='cuda:1'):
        decoder.group_objects(depth, centers, decoder.extract_peaks(heat), cameras=other)
    with pytest.raises(ValueError, match='cuda:1'):
        decoder.decode_host_batch(*(t.cpu() for t in (heat, depth, centers)), cameras=other)


@gpu
@pytest.mark.parametrize('dtype', ['bf16', 'f16'])
def test_mixed_map_types_take_the_two_call_path_with_the_table(dtype):
    """16-bit heatmaps with float32 depth / centre maps: okp_extract_peaks_* then okp_group_objects_cameras_f32."""
    from oracle import c_oracle
    from object_keypoints_b200 import KeypointDecoder
    size = (64, 64)
    cameras = _cameras(size)
    heat32, depth, centers = (t.cuda() for t in _batch(size))
    heat = heat32.to(DTYPES[dtype])
    index = _index('random', heat.shape[0])
    decoder = KeypointDecoder(CFG, size)
    got = decoder.decode_batch(heat, depth, centers, cameras=decoder.camera_table(cameras, index)).numpy()
    for c, camera in enumerate(cameras):
        idx = np.flatnonzero(index == c)
        want = c_oracle.decode(heat.float().cpu().numpy()[idx], depth.cpu().numpy()[idx], centers.cpu().numpy()[idx], CFG, camera)
        assert_matches_oracle(_rows(got, idx, False), want)


def _records(decoder, maps, N, cameras=None):
    buffer = torch.zeros((N, decoder.record_bytes()), dtype=torch.uint8, device='cuda')
    pointers = (ctypes.c_void_p * 1)(buffer.data_ptr())
    sink = _abi.OkpRecordSink(buffers_dev=pointers, n_buffers=1, record_bytes=decoder.record_bytes(), first_row=0)
    decoder.decode_batch(*maps, records=sink, cameras=cameras)
    torch.cuda.synchronize()
    return buffer.cpu()


@gpu
@pytest.mark.parametrize('dtype', ['f32', 'bf16', 'f16'])
@pytest.mark.parametrize('size', [(180, 320), (64, 64)])
def test_records_are_those_of_the_single_camera_decodes(size, dtype):
    from object_keypoints_b200 import KeypointDecoder
    cameras = _cameras(size)
    maps, _ = _maps(size, dtype)
    N = maps[0].shape[0]
    index = _index('random', N)
    decoder = KeypointDecoder(CFG, size)
    got = _records(decoder, maps, N, decoder.camera_table(cameras, index))
    want = torch.zeros_like(got)
    for c, camera in enumerate(cameras):
        idx = np.flatnonzero(index == c)
        sel = torch.from_numpy(idx).cuda()
        want[torch.from_numpy(idx)] = _records(KeypointDecoder(CFG, size, camera=camera), [m[sel] for m in maps], idx.size)
    assert torch.equal(got, want)
    assert got.view(torch.int32)[:, 0].sum() > 0


@gpu
@pytest.mark.parametrize('dtype,sparse', [('f32', 'only'), ('bf16', False)])
def test_host_batch_reads_each_chunks_rows_of_the_table(dtype, sparse):
    """chunk_frames 7 against camera blocks of 5 frames: chunks start in the middle of a block."""
    from object_keypoints_b200 import KeypointDecoder
    size = (64, 64)
    cameras = _cameras(size)
    host = [t[:37].to(DTYPES[dtype]).contiguous() for t in _batch(size)]
    index = (np.arange(37) // 5) % 3
    decoder = KeypointDecoder(CFG, size)
    table = decoder.camera_table(cameras, index)
    want = decoder.decode_batch(*(t.cuda() for t in host), cameras=table).numpy()
    for pinned in (True, False):
        inputs = [t.pin_memory() for t in host] if pinned else host
        got = decoder.decode_host_batch(*inputs, chunk_frames=7, sparse=sparse, cameras=table)
        for name in KeypointDecoder.HOST_RESULT_TABLES:
            np.testing.assert_array_equal(got[name].numpy().view(np.uint8), want[name].view(np.uint8), err_msg=f"{pinned} {name}")
        assert (decoder.host_chunks_sparse > 0) == (sparse == 'only')
    with pytest.raises(ValueError, match='rows'):
        decoder.decode_host_batch(*(t[:36] for t in host), chunk_frames=7, cameras=table)


# ---------------------------------------------------------------------------------------------------------------------
# Stereo scene: both views of a rig decoded in one call
# ---------------------------------------------------------------------------------------------------------------------
STEREO_SIZE, STEREO_CFG, STEREO_PAIRS = (180, 320), [1, 1, 1], 8


def _stereo_scene():
    """Three objects (a centre and three keypoints each) per pair, 0.7-1.1 m in front of cam0, left of the image column
    the reference's clip (compat_clip_bug: x clipped with H - 1) would move. -> keypoints [2P, 3, 4, 2] and depths
    [2P, 3, 4] in prediction pixels / metres, rows left, right, left, ...; cam0, cam1 at the prediction size; T_LR."""
    cam0, cam1, p = _rig()
    cam0, cam1 = _fit(cam0, STEREO_SIZE), _fit(cam1, STEREO_SIZE)
    keypoints, depths = [], []
    for pair in range(STEREO_PAIRS):
        rng = np.random.default_rng(100 + pair)
        X = []
        for g in range(3):
            z = rng.uniform(0.7, 1.1)
            c = np.array([(-0.3 + 0.16 * g + rng.uniform(-0.02, 0.02)) * z, rng.uniform(-0.2, 0.2) * z, z])
            angles = rng.uniform(0, 2 * np.pi) + np.arange(3) * 2 * np.pi / 3
            X.append([c] + [c + 0.05 * np.array([np.cos(a), np.sin(a), 0.2 * rng.uniform(-1, 1)]) for a in angles])
        X = np.array(X).reshape(-1, 3)
        for camera, T in ((cam0, np.eye(4)), (cam1, p['T_RL'])):
            keypoints.append(camera.project(X, T).reshape(3, 4, 2))
            depths.append((X @ T[:3, :3].T + T[:3, 3])[:, 2].reshape(3, 4))
    return np.array(keypoints), np.array(depths), cam0, cam1, p['T_LR']


def _stereo_error(tables, T_LR):
    """Largest distance between a left-view point and the right-view point of the same object mapped by T_LR (objects
    matched by their nearest mapped centre)."""
    worst = 0.0
    for pair in range(STEREO_PAIRS):
        left, right = 2 * pair, 2 * pair + 1
        assert tables['n_objects'][left] == tables['n_objects'][right] == 3
        assert (tables['kp_count'][[left, right], :3] == 1).all()
        mapped = tables['kp_point'][right, :3, :, 0] @ T_LR[:3, :3].T + T_LR[:3, 3]          # [3, C, 3]
        for o in range(3):
            own = tables['kp_point'][left, o, :, 0]
            r = np.argmin(np.linalg.norm(mapped[:, 0] - own[0], axis=1))
            worst = max(worst, float(np.abs(mapped[r] - own).max()))
    return worst


def test_stereo_tolerance_on_the_oracle():
    """The CPU rehearsal behind STEREO_TOL: the C oracle decodes each view with its own camera (within the tolerance)
    and with cam0 for both views (outside it)."""
    from oracle import c_oracle, np_oracle
    keypoints, depths, cam0, cam1, T_LR = _stereo_scene()
    maps = [np_oracle.rasterise_targets(k, d, STEREO_CFG, STEREO_SIZE) for k, d in zip(keypoints, depths)]
    heat, centers, depth = (np.array([m[i] for m in maps]) for i in range(3))
    left_model = c_oracle.decode(heat, depth, centers, STEREO_CFG, cam0)
    own = {k: v.copy() for k, v in left_model.items()}
    own['kp_point'][1::2] = c_oracle.decode(heat, depth, centers, STEREO_CFG, cam1)['kp_point'][1::2]
    assert _stereo_error(own, T_LR) < STEREO_TOL < _stereo_error(left_model, T_LR)


@gpu
def test_stereo_pairs_decode_in_one_call_with_each_views_camera():
    from object_keypoints_b200 import KeypointDecoder, targets
    keypoints, depths, cam0, cam1, T_LR = _stereo_scene()
    heat, depth, centers = targets.rasterise_targets(keypoints, depths, STEREO_CFG, STEREO_SIZE)
    decoder = KeypointDecoder(STEREO_CFG, STEREO_SIZE, camera=cam0)
    table = decoder.camera_table((cam0, cam1), np.arange(2 * STEREO_PAIRS) % 2)
    stereo = decoder.decode_batch(heat, depth, centers, cameras=table).numpy()
    assert _stereo_error(stereo, T_LR) < STEREO_TOL
    # the same batch lifted with cam0 alone: nothing fails, the right views' points are off
    assert _stereo_error(decoder.decode_batch(heat, depth, centers).numpy(), T_LR) > STEREO_TOL


# ---------------------------------------------------------------------------------------------------------------------
# Host checks (no GPU)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('size', [(180, 320), (64, 64)])
def test_camera_recipe_is_the_default_camera(size):
    from object_keypoints_b200 import synthetic
    assert bytes(_abi.pack_camera(_cameras(size)[0])) == bytes(_abi.pack_camera(synthetic.default_camera(size)))


def test_pack_camera_table_rows_are_pack_camera():
    cameras = _cameras((64, 64))
    packed = [bytes(_abi.pack_camera(c)) for c in cameras]
    assert len(set(packed)) == 3 and len({(_abi.pack_camera(c).clip_x, _abi.pack_camera(c).clip_y) for c in cameras}) == 2
    for index in ([2, 0, 1, 1, 0, 2, 2], np.array([1], np.uint8), np.arange(12) % 3, []):
        table = _abi.pack_camera_table(cameras, index)
        assert len(table) == len(index)
        assert ctypes.sizeof(table) == 144 * len(index)
        for n, c in enumerate(np.asarray(index).tolist()):
            assert bytes(table[n]) == packed[c]


@pytest.mark.parametrize('index,match', [
    ([0, 3], 'range'), ([0, -1], 'range'), (np.array([0.0, 1.0]), 'integers'), ([0, 1.5], 'integers'),
    ([True, False], 'integers'), (np.zeros((2, 2), np.int64), '1-D'), (1, '1-D'),
])
def test_pack_camera_table_rejects_bad_indices(index, match):
    with pytest.raises(ValueError, match=match):
        _abi.pack_camera_table(_cameras((64, 64)), index)


def test_camera_entries_validate_their_arguments_on_the_host():
    """NULL table or depth, a misaligned table and single_pass are refused before anything touches a device (the other
    pointers are never dereferenced)."""
    if _lib.needs_build():
        _lib.build()
    lib = _lib.lib()
    tables, cfg = _abi.OkpDecodeTables(), (ctypes.c_int32 * 2)(1, 3)
    fake = ctypes.c_void_p(1 << 20)
    aligned, misaligned = ctypes.c_void_p(1 << 21), ctypes.c_void_p((1 << 21) + 8)
    prm, single = _abi.make_params(), _abi.make_params(single_pass=True)
    for suffix in ('f32', 'bf16', 'f16'):
        decode = getattr(lib, f'okp_decode_cameras_{suffix}')
        group = getattr(lib, f'okp_group_objects_cameras_{suffix}')

        def calls(depth, cameras, p):
            yield decode(fake, depth, fake, 4, 3, 64, 64, cfg, cameras, ctypes.byref(p), ctypes.byref(tables), fake, 1 << 20,
                         None, None)
            yield group(depth, fake, 4, 3, 64, 64, cfg, cameras, ctypes.byref(p), ctypes.byref(tables), None, None)

        assert set(calls(fake, None, prm)) == {-1}, suffix             # OKP_E_NULL
        assert set(calls(None, aligned, prm)) == {-1}, suffix
        assert set(calls(fake, misaligned, prm)) == {-4}, suffix       # OKP_E_UNSUPPORTED
        assert set(calls(fake, aligned, single)) == {-4}, suffix
        # no frames: OKP_OK whatever the pointers, like every other entry
        assert decode(None, None, None, 0, 3, 64, 64, cfg, None, ctypes.byref(prm), ctypes.byref(tables), None, 0, None,
                      None) == 0, suffix
        assert group(None, None, 0, 3, 64, 64, cfg, None, ctypes.byref(prm), ctypes.byref(tables), None, None) == 0, suffix
